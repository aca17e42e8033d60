"""The IDM traffic model of the rollouts (include/pp.h, PP_TRAFFIC_IDM) on the CPU: the
restatement in traffic_oracle.c driven with scripted scenarios on a straight road (and, for the
loop seam, on the highway map).  The GPU side is checked against this restatement in
test_traffic.py.

In these scenarios the planner is not in the loop: every plan is empty (the ego stays where it is
and dt = 0.02 s) and reports every car in its lane at s = 0, so no car is respawned."""
import numpy as np
import pytest

import checkers
import traffic_oracle

abi = checkers.abi
SEG = 30.0  # waypoint spacing of the straight road
LANE_Y = [-2.0, -6.0, -10.0]  # lane centres: the reference line is y = 0, d grows to the right
HALF_LEN = 4.5  # PP_INC_CAR_HALF_LEN


@pytest.fixture(scope="module")
def road():
    """The model on a straight road along +x (the scenarios stay far from its wrap-around)."""
    n = 800
    return traffic_oracle.TrafficOracle(points=(SEG * np.arange(n), np.zeros(n)))


def scene(pp, tor, cars, ego=(2, 100.0)):
    """One rollout on the straight road: cars [(lane, x, v, v0)], the ego at rest at (lane, x)
    (or at (d, x) when the first entry is a float: d metres right of the reference line)."""
    st = pp.RolloutStateHost(1, len(cars))
    for j, (lane, x, v, _) in enumerate(cars):
        w = int(x // SEG) + 1
        st.car_lane[0, j] = lane
        st.car_wp[0, j] = w
        st.car_ratio[0, j] = (x - SEG * (w - 1)) / SEG
        st.car_speed[0, j] = v
    st.ego_x[0] = ego[1]
    st.ego_y[0] = -ego[0] if isinstance(ego[0], float) else LANE_Y[ego[0]]
    ts = tor.init(st)
    ts["car_v0"][0, :] = [v0 for *_, v0 in cars]
    return st, ts


def tick(tor, st, ts):
    pb = abi.PlanBatch(1, max(st.n_cars, 1), diag=False, cars=True)
    pb.n_points[0] = 0
    pb.ref_wp[0] = int(st.ego_x[0] // SEG) + 1
    pb.car_lane[0, :st.n_cars] = st.car_lane[0]
    pb.car_s[0, :st.n_cars] = 0.0
    tor.advance(st, ts, 0, 0, 1, pb)


def car_x(st, j):
    return SEG * (st.car_wp[0, j] - 1) + st.car_ratio[0, j] * SEG


def run(tor, st, ts, ticks, pin=()):
    """ticks ticks; the cars in `pin` are put back where they were, at rest, after every tick.
    Returns x [ticks + 1][C], v [ticks + 1][C], acc [ticks][C]."""
    keep = {j: (st.car_wp[0, j], st.car_ratio[0, j]) for j in pin}
    xs = [[car_x(st, j) for j in range(st.n_cars)]]
    vs = [st.car_speed[0].copy()]
    accs = []
    for _ in range(ticks):
        tick(tor, st, ts)
        for j, (w, u) in keep.items():
            st.car_wp[0, j], st.car_ratio[0, j], st.car_speed[0, j] = w, u, 0.0
        xs.append([car_x(st, j) for j in range(st.n_cars)])
        vs.append(st.car_speed[0].copy())
        accs.append(ts["car_acc"][0].copy())
    return np.array(xs), np.array(vs), np.array(accs)


def idm_acc(v, v0, delta=None, vl=0.0):
    """pp.h's formula in the same operations, for exact comparisons."""
    q = v / v0
    q2 = q * q
    inter = 0.0
    if delta is not None:
        gap = max(delta - HALF_LEN, abi.TRF_GAP_FLOOR)
        dyn = max(v * abi.TRF_HEADWAY + v * (v - vl) / (2.0 * np.sqrt(abi.TRF_ACC * abi.TRF_DEC)), 0.0)
        z = (abi.TRF_MIN_GAP + dyn) / gap
        inter = z * z
    acc = abi.TRF_ACC * (1.0 - q2 * q2 - inter)
    return min(max(acc, -abi.TRF_MAX_DEC), abi.TRF_ACC)


def test_free_road(pp, road):
    st, ts = scene(pp, road, [(1, 600.0, 0.0, 20.0)])
    _, v, acc = run(road, st, ts, 2500)
    v = v[:, 0]
    assert (np.diff(v) >= 0).all() and v.max() <= 20.0
    assert v[-1] > 19.9
    assert acc[0, 0] == abi.TRF_ACC and (acc <= abi.TRF_ACC).all()


def test_stopped_leader(pp, road):
    st, ts = scene(pp, road, [(1, 600.0, 20.0, 20.0), (1, 800.0, 0.0, 20.0)])
    x, v, acc = run(road, st, ts, 3000, pin=(1,))
    gap = x[:, 1] - x[:, 0] - HALF_LEN
    assert (gap > 0).all() and (v[:, 0] >= 0).all()
    assert v[-1, 0] < 1e-3
    # the restatement's follower comes to rest at tick 832 with a gap of 1.9407 m and stays
    # there: the 0.02 s explicit step overshoots s0 = 2 m by 6 cm before the speed floor holds it;
    # 0.1 m is that overshoot with room for rounding, not for a different trajectory
    assert abs(gap[-1] - abi.TRF_MIN_GAP) < 0.1, gap[-1]
    assert acc.min() >= -abi.TRF_MAX_DEC


def test_platoon_settles_behind_a_slow_leader(pp, road):
    cars = [(1, 1000.0, 15.0, 15.0)] + [(1, 1000.0 - 30.0 * i, 20.0, 25.0) for i in range(1, 7)]
    st, ts = scene(pp, road, cars)
    x, v, acc = run(road, st, ts, 6000)
    assert (np.diff(x, axis=1) < -HALF_LEN).all()  # in order, no overlap, at every tick
    assert np.abs(v[-1] - 15.0).max() < 0.01, v[-1]
    assert (v[:, 0] == 15.0).all() and (acc[:, 0] == 0.0).all()
    assert (v <= 25.0).all() and (v >= 0).all()


def test_the_ego_leads(pp, road):
    # a car behind the ego at rest in lane 1 stops behind it; one in lane 0 passes
    st, ts = scene(pp, road, [(1, 600.0, 20.0, 20.0), (0, 600.0, 20.0, 20.0)], ego=(1, 750.0))
    assert ts["ego_lanes"][0] == 0b010
    x, v, _ = run(road, st, ts, 3000)
    gap = 750.0 - x[:, 0] - HALF_LEN
    assert (gap > 0).all() and v[-1, 0] < 1e-3 and abs(gap[-1] - abi.TRF_MIN_GAP) < 0.1  # 1.9406 m
    assert x[-1, 1] > 750.0 + 500.0 and v[-1, 1] > 19.9
    # the ego at d = 8, between lanes 1 and 2, leads both
    st, ts = scene(pp, road, [(0, 600.0, 20.0, 20.0)], ego=(8.0, 750.0))
    assert ts["ego_lanes"][0] == 0b110


def test_loop_seam(pp, oracle):
    tor = traffic_oracle.TrafficOracle()
    n = tor.n_wp
    st = pp.RolloutStateHost(1, 2)
    st.car_lane[0] = 1
    st.car_wp[0] = [n - 1, 1]  # follower just before the last waypoint, leader past waypoint 0
    st.car_ratio[0] = [0.5, 0.5]
    st.car_speed[0] = [20.0, 5.0]
    tbl = oracle.map_table()
    st.ego_x[0], st.ego_y[0] = tbl[90, 6], tbl[90, 7]  # lane 2, far away
    ts = tor.init(st)
    assert ts["ego_lanes"][0] == 0b100
    cum = tor.cum[1]
    s = [cum[n - 1] + 0.5 * tbl[n - 1, 11], cum[1] + 0.5 * tbl[1, 11]]
    delta = s[1] - s[0] + cum[n]
    assert 0 < delta < 100.0
    pb = abi.PlanBatch(1, 2, diag=False, cars=True)
    pb.ref_wp[0] = 90
    pb.car_lane[0] = 1
    tor.advance(st, ts, 0, 0, 1, pb)
    want = idm_acc(20.0, 20.0, delta, 5.0)
    assert ts["car_acc"][0, 0] == want and want < -1.0
    assert ts["car_acc"][0, 1] == idm_acc(5.0, 5.0)  # the follower is behind the leader, not ahead
    assert st.car_wp[0, 0] in (n - 1, 0)


def test_equal_s_is_decided_by_the_slot(pp, road):
    st, ts = scene(pp, road, [(1, 600.0, 20.0, 25.0), (1, 600.0, 20.0, 25.0)])
    tick(road, st, ts)
    acc = ts["car_acc"][0]
    assert acc[0] == -abi.TRF_MAX_DEC  # slot 1 is ahead of slot 0: the gap floor
    assert acc[1] == idm_acc(20.0, 25.0)  # slot 0 is not ahead of slot 1: free road
    assert np.isfinite(st.car_speed).all() and np.isfinite(st.car_ratio).all()


def test_overlapping_placement_brakes_at_the_clamp(pp, road):
    st, ts = scene(pp, road, [(1, 600.0, 1.0, 20.0), (1, 602.0, 0.0, 20.0)])
    x, v, acc = run(road, st, ts, 50, pin=(1,))
    assert (acc[:, 0] == -abi.TRF_MAX_DEC).all()
    assert (v[:, 0] >= 0).all() and v[-1, 0] == 0.0
    assert v[1, 0] == 1.0 - abi.TRF_MAX_DEC * 0.02
