"""The episode restarts of the rollouts (include/pp.h, pp_rollouts_set_restart) on the CPU: the
restatement in restart_oracle.c, after the monitor's, driven with scripted points and cars on a
straight road, where every expectation is exact.  The GPU side is checked against this
restatement in test_restarts.py.

One rollout; each tick drives one point (k = 1), and the cars are static unless a scenario moves
them, so a collision begins when the ego drives into a car."""
import numpy as np
import pytest

import checkers
import restart_oracle

abi = checkers.abi
INC = abi.INC
NONFINITE = abi.REC_NONFINITE
SEG = 30.0  # waypoint spacing of the straight road
LANE_Y = [-2.0, -6.0, -10.0]  # lane centres: the reference line is y = 0, d grows to the right
SEED, FIRST = 99, 7
M64 = (1 << 64) - 1


def mix64(z):
    """splitmix64, as pp.h states it."""
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def key(seed, rollout, e):
    k0 = mix64(mix64(seed ^ 0x1417) ^ ((rollout * 0xD1B54A32D192ED03) & M64))
    return k0 if e == 0 else mix64((k0 + e * 0xA0761D6478BD642F) & M64)


@pytest.fixture(scope="module")
def road():
    n = 800
    return restart_oracle.RestartOracle(points=(SEG * np.arange(n), np.zeros(n)))


class Sim:
    """One rollout on the straight road: the ego at (x, lane centre) with `cars` [(lane, x)]."""

    def __init__(self, pp, ro, mask, cars=(), x=600.0, lane=1, idm=False):
        self.pp, self.ro, self.mask, self.c = pp, ro, mask, len(cars)
        st = pp.RolloutStateHost(1, self.c)
        st.ego_x[0], st.ego_y[0], st.target_lane[0] = x, LANE_Y[lane], lane
        self.place(st, cars)
        self.st = st
        self.ms = ro.monitor.init(st.ego_x, st.ego_y)
        self.ts = ro.traffic.init(st) if idm else None
        self.rs = ro.init(1)

    @staticmethod
    def place(st, cars):
        for j, (lane, x) in enumerate(cars):
            w = int(x // SEG) + 1
            st.car_lane[0, j], st.car_wp[0, j] = lane, w
            st.car_ratio[0, j] = (x - SEG * (w - 1)) / SEG
            st.car_speed[0, j] = 20.0

    def tick(self, dx=0.4, point=None, cars_after=None):
        st, mc = self.st, max(self.c, 1)
        fb = abi.FrameBatch(1, mc)
        fb.ego_x[0], fb.ego_y[0] = st.ego_x[0], st.ego_y[0]
        px, py = point if point is not None else (st.ego_x[0] + dx, st.ego_y[0])
        pb = abi.PlanBatch(1, mc, diag=False, cars=False)
        pb.n_points[0] = abi.PATH_LEN
        pb.next_x[0, 0], pb.next_y[0, 0] = px, py
        pb.ref_wp[0] = int((px if np.isfinite(px) else st.ego_x[0]) // SEG) + 1
        before = restart_oracle_copy(self.pp, st)
        after = restart_oracle_copy(self.pp, st)
        if cars_after is not None:
            self.place(after, cars_after)
        self.ro.monitor.step(self.ms, self.c, 1, fb, pb, before, after)
        for k in ("car_lane", "car_wp", "car_ratio", "car_speed"):
            getattr(st, k)[...] = getattr(after, k)
        st.ego_x[0], st.ego_y[0] = px, py
        st.tick += 1
        self.ro.step(self.rs, st, self.ms, self.ts, self.c, SEED, FIRST, self.mask)
        return {k: v[0].copy() for k, v in self.rs.rec.items()}

    def inc(self, name):
        return int(self.ms.rec["count"][0, INC[name]])


def restart_oracle_copy(pp, st):
    out = pp.RolloutStateHost(st.n, st.n_cars)
    for name, _, _ in abi.ROLLOUT_STATE_FIELDS:
        getattr(out, name)[...] = getattr(st, name)
    out.tick = st.tick
    return out


def assert_fresh_episode(sim, e, tick, dist):
    """The rollout restarted into episode e at `tick` after driving `dist` in all."""
    st, ms, rec = sim.st, sim.ms, sim.rs.rec
    want = sim.ro.draw(sim.pp, SEED, FIRST, 1, sim.c, episodes=[e])
    for name, _, _ in abi.ROLLOUT_STATE_FIELDS:
        assert np.array_equal(getattr(st, name), getattr(want, name)), name
    assert st.ego_speed_mph[0] == 0.0 and st.path_n[0] == 0
    assert rec["episodes"][0] == e and rec["episode_tick"][0] == tick
    assert rec["episode_m"][0] == dist == ms.rec["distance_m"][0]
    assert ms.pts[0] == 0 and ms.active[0] == 0 and ms.off_pts[0] == 0
    assert ms.rec["clean_m"][0] == 0.0
    assert ms.ring[0, 0, 0] == st.ego_x[0] and ms.ring[0, 0, 1] == st.ego_y[0]


def test_keys_follow_the_stated_rule(road):
    for r in (0, 1, 12345):
        for e in (0, 1, 2, 3, 1000):
            assert road.key(SEED, r, e) == key(SEED, r, e), (r, e)


def test_front_collision_restarts_into_episode_1(pp, road):
    sim = Sim(pp, road, ["collision_front"], cars=[(1, 606.5)])
    hit = None
    for t in range(20):
        rec = sim.tick()
        if rec["episodes"]:
            hit = t
            break
    assert hit is not None and sim.inc("collision_front") == 1
    d = sim.ms.rec["distance_m"][0]
    assert d > 0
    assert rec["by_bit"][INC["collision_front"]] == 1 and rec["by_bit"].sum() == 1
    assert rec["ended_m"] == d and rec["ended_lap"] == 0
    assert_fresh_episode(sim, 1, hit + 1, d)
    # the next episode drives on: distance keeps growing from there, no further restart
    for _ in range(30):
        rec = sim.tick()
    assert rec["episodes"] == 1 and sim.ms.rec["distance_m"][0] > d
    assert sim.ms.rec["first_tick"][0] == hit and sim.ms.rec["count"][0].sum() >= 1


@pytest.mark.parametrize("with_rear", [False, True])
def test_rear_collision_restarts_only_with_its_bit(pp, road, with_rear):
    mask = ["collision_front"] + (["collision_rear"] if with_rear else [])
    sim = Sim(pp, road, mask, cars=[(1, 590.0)])
    rec = None
    for t in range(20):
        rec = sim.tick(cars_after=[(1, 590.0 + 0.9 * (t + 1))])
        if sim.inc("collision_rear"):
            break
    assert sim.inc("collision_rear") == 1 and sim.inc("collision_front") == 0
    if with_rear:
        assert rec["episodes"] == 1 and rec["by_bit"][INC["collision_rear"]] == 1
        assert_fresh_episode(sim, 1, t + 1, sim.ms.rec["distance_m"][0])
    else:
        assert rec["episodes"] == 0 and rec["by_bit"].sum() == 0
        assert sim.st.ego_y[0] == LANE_Y[1] and sim.st.ego_x[0] > 600.0  # still driving on


@pytest.mark.parametrize("mask,bit", [(["nonfinite"], NONFINITE),
                                      (["off_road", "nonfinite"], INC["off_road"])])
def test_nan_plan_restarts_with_the_distance_restored(pp, road, mask, bit):
    sim = Sim(pp, road, mask)
    for _ in range(5):
        sim.tick()
    d = sim.ms.rec["distance_m"][0]
    rec = sim.tick(point=(np.nan, np.nan))
    assert sim.inc("off_road") == 1  # the NaN point is also off the road, in the same tick
    assert rec["episodes"] == 1 and rec["by_bit"][bit] == 1 and rec["by_bit"].sum() == 1
    assert sim.ms.rec["distance_m"][0] == d == rec["ended_m"]
    assert_fresh_episode(sim, 1, 6, d)
    for _ in range(20):  # a restored distance does not fire again
        rec = sim.tick()
    assert rec["episodes"] == 1 and np.isfinite(sim.ms.rec["distance_m"][0])


def test_nan_without_its_bit_stays_nan(pp, road):
    sim = Sim(pp, road, ["collision_front"])
    sim.tick()
    rec = sim.tick(point=(np.nan, np.nan))
    assert rec["episodes"] == 0 and np.isnan(sim.ms.rec["distance_m"][0])


def test_idm_state_is_reset(pp, road):
    sim = Sim(pp, road, ["collision_front"], cars=[(1, 606.5), (0, 650.0), (2, 700.0)], idm=True)
    sim.ts["car_v0"][0] = [25.0, 26.0, 27.0]
    sim.ts["car_acc"][0] = [-1.0, 0.5, 1.5]
    for _ in range(20):
        rec = sim.tick()
        if rec["episodes"]:
            break
    assert rec["episodes"] == 1
    want = road.traffic.init(sim.st)
    for k in want.arrays:
        assert np.array_equal(sim.ts[k], want[k]), k
    assert np.array_equal(sim.ts["car_v0"], sim.st.car_speed) and (sim.ts["car_acc"] == 0).all()


def test_episode_2_uses_key_2(pp, road):
    sim = Sim(pp, road, ["nonfinite"])
    sim.tick()
    sim.tick(point=(np.nan, np.nan))
    sim.tick()
    d = sim.ms.rec["distance_m"][0]
    rec = sim.tick(point=(np.nan, np.nan))
    assert rec["episodes"] == 2 and rec["by_bit"][NONFINITE] == 2
    assert rec["episode_tick"] == 4 and rec["ended_m"] == d
    assert_fresh_episode(sim, 2, 4, d)
    assert road.key(SEED, FIRST, 2) == key(SEED, FIRST, 2) != key(SEED, FIRST, 1)


@pytest.mark.parametrize("below", [False, True])
def test_ended_lap_at_exactly_the_rubric(pp, road, below):
    sim = Sim(pp, road, ["over_speed"])
    lap = abi.RST_RUBRIC_M
    assert lap == 4.32 * 1609.344
    d = np.nextafter(lap, 0.0) if below else lap
    # the monitor's record as if the episode had driven d and counted an over-speed in this tick
    sim.ms.rec["distance_m"][0] = d
    sim.ms.rec["count"][0, INC["over_speed"]] = 1
    road.step(sim.rs, sim.st, sim.ms, None, 0, SEED, FIRST, sim.mask)
    rec = sim.rs.rec
    assert rec["episodes"][0] == 1 and rec["ended_m"][0] == d
    assert rec["ended_lap"][0] == (0 if below else 1)
