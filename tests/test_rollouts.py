"""Closed-loop rollouts (BASELINE config 3, SURVEY §8f-1).

GPU: every tick of pp_rollouts_run is checked three ways against the CPU
checker — the frame the device simulator produced (bit-exact), the plan for that
frame (teacher-forced: same inputs; integers and + - * / quantities bit-exact,
trajectories within 1e-9 rel / 1e-6 m), and the simulator's next state given the
device's plan (bit-exact) — for consume_k = 1 and 3, then a free-running
comparison (CPU loop vs device loop from the same initial state) reports the
divergence.
CPU: the simulator model itself on the oracle planner (sanity of the model).
"""
import copy
import os

import numpy as np
import pytest

import checkers

INT_FIELDS = ("n_points", "ego_lane", "ref_wp", "target_lane", "flags", "car_lane", "car_next_wp",
              "next_car_id", "next_car_in_target_lane")
EXACT_FIELDS = ("ego_s", "ego_d", "ego_vs", "ego_vd", "ego_speed", "ego_acc", "target_speed",
                "target_time", "car_s", "car_d", "car_vs", "car_vd")
STATE_FIELDS = [n for n, _, _ in checkers.abi.ROLLOUT_STATE_FIELDS]


def assert_plans_match(got, want, where):
    for k in INT_FIELDS:
        assert np.array_equal(getattr(got, k), getattr(want, k)), (where, k)
    for k in EXACT_FIELDS:
        assert np.array_equal(getattr(got, k), getattr(want, k), equal_nan=True), (where, k)
    for k in ("next_x", "next_y"):
        a, b = getattr(got, k), getattr(want, k)
        assert np.array_equal(a != a, b != b), (where, k)
        err = np.nanmax(np.abs(a - b))
        rel = np.nanmax(np.abs(a - b) / np.maximum(np.abs(b), 1.0))
        assert err <= 1e-6 and rel <= 1e-9, (where, k, err, rel)


def cpu_state_from(pp, st):
    out = pp.RolloutStateHost(st.n, st.n_cars)
    for k in STATE_FIELDS:
        getattr(out, k)[...] = getattr(st, k)
    out.tick = st.tick
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name", ["default", "loose", "max25"])
@pytest.mark.parametrize("consume_k", [1, 3])
def test_rollout_ticks_match_cpu_model_and_planner(pp, oracle, consume_k, cfg_name):
    """Planner tunables reach the planning step of the loop: `loose` (max_speed 40, hard
    acceleration) is where the ego drives at 30-40 m/s, speeds no synthetic frame has."""
    cfg = checkers.config(cfg_name)
    n, c, seed, first, ticks = 192, 12, 77, 1000, 60
    m = pp.Map()
    ro = pp.Rollouts(m, n, c, seed=seed, first=first)
    prev = ro.state()
    assert prev.tick == 0 and (prev.path_n == 0).all()
    respawns, top_speed = 0, 0.0
    for t in range(ticks):
        ro.run(1, consume_k, cfg=cfg)
        frames, plans = ro.last()
        now = ro.state()
        # 1. the frame the device simulator built from the previous state
        want_frames = oracle.sim_frames(prev, c)
        for k, a in frames.arrays().items():
            assert np.array_equal(a, getattr(want_frames, k)), (t, k)
        # 2. the plan for that frame (teacher-forced)
        assert_plans_match(plans, oracle.plan(frames, threads=4, cfg=cfg), t)
        top_speed = max(top_speed, float(plans.ego_speed.max()))
        # 3. the simulator step given the device's plan
        cpu = cpu_state_from(pp, prev)
        oracle.sim_advance(cpu, c, seed, first, consume_k, plans)
        for k in STATE_FIELDS:
            assert np.array_equal(getattr(now, k), getattr(cpu, k)), (t, k)
        assert now.tick == cpu.tick == t + 1
        respawns += int(((plans.car_lane < 0) | (plans.car_s < -100) | (plans.car_s > 300)).sum())
        prev = now
    assert (prev.path_n == 50 - consume_k).all()
    # the loop actually drives: the ego moved, traffic was recycled
    first_state = pp.Rollouts(m, n, c, seed=seed, first=first).state()
    moved = np.hypot(prev.ego_x - first_state.ego_x, prev.ego_y - first_state.ego_y)
    assert moved.min() > 0.5 and respawns > 0
    if cfg_name == "loose":
        assert top_speed > 30.0
    stats = ro.stats().cpu().numpy()
    assert stats[0] == n * ticks and stats[1] == 50 * n * ticks


@pytest.mark.gpu
def test_rollout_groups_and_graph_replay_match_cpu_model(pp, oracle):
    """Enough rollouts for several stream groups, enough ticks for the captured-graph path:
    the device state after T ticks equals tick-by-tick stepping of a second, identical job,
    and the last tick is checked against the CPU planner and model."""
    n, c, seed, ticks, k = 12288, 12, 21, 12, 2
    m = pp.Map()
    a = pp.Rollouts(m, n, c, seed=seed)
    b = pp.Rollouts(m, n, c, seed=seed)
    a.set_groups(3)  # three stream groups of 4,096; b: automatic (one group at this size)
    os.environ["PP_ROLLOUT_GRAPH"] = "1"
    try:
        a.run(ticks, k)        # >= 8 ticks: one direct tick, then graph replays
    finally:
        del os.environ["PP_ROLLOUT_GRAPH"]
    for _ in range(ticks):
        b.run(1, k)            # direct issue
    sa, sb = a.state(), b.state()
    for f in STATE_FIELDS:
        assert np.array_equal(getattr(sa, f), getattr(sb, f)), f
    assert sa.tick == sb.tick == ticks
    assert np.array_equal(a.stats().cpu().numpy(), b.stats().cpu().numpy())
    # one more tick, checked on the CPU
    prev = sa
    a.run(1, k)
    frames, plans = a.last()
    want_frames = oracle.sim_frames(prev, c)
    for key, arr in frames.arrays().items():
        assert np.array_equal(arr, getattr(want_frames, key)), key
    assert_plans_match(plans, oracle.plan(frames, threads=8), "tick %d" % ticks)
    cpu = cpu_state_from(pp, prev)
    oracle.sim_advance(cpu, c, seed, 0, k, plans)
    now = a.state()
    for f in STATE_FIELDS:
        assert np.array_equal(getattr(now, f), getattr(cpu, f)), f


@pytest.mark.gpu
@pytest.mark.parametrize("n", [700, 6000])
def test_rollout_statistics_are_the_sum_of_the_ticks(pp, n):
    """pp_rollouts_stats == sum over the ticks of pp_stats_batch over that tick's plans, every
    entry, the trajectory checksum included — for a job small enough for the single-kernel
    planner (the simulator kernel takes the checksum) and for one on the pipeline (the planning
    kernels add it as they write the points)."""
    import torch
    c, ticks, k = 12, 5, 2
    m = pp.Map()
    ro = pp.Rollouts(m, n, c, seed=5)
    want = np.zeros(pp.STATS_LEN, dtype=np.int64)
    for _ in range(ticks):
        ro.run(1, k)
        _, plans = ro.last()
        dp = pp.DevicePlans(n, max(c, 1), diag=False, cars=False)
        for name in dp.t:
            a = getattr(plans, name)
            dp.t[name].copy_(torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a))
        want += pp.stats_batch(dp).cpu().numpy()
    got = ro.stats().cpu().numpy()
    assert np.array_equal(got, want), (got, want)
    assert got[pp.abi.STAT_XSUM] != 0


@pytest.mark.gpu
def test_rollout_free_running_divergence(pp, oracle):
    """Device loop vs CPU loop, each feeding back its OWN plans, from the same initial state."""
    n, c, seed, ticks, k = 128, 12, 5, 150, 2
    m = pp.Map()
    ro = pp.Rollouts(m, n, c, seed=seed)
    cpu = cpu_state_from(pp, ro.state())
    ro.run(ticks, k)
    gpu = ro.state()
    for _ in range(ticks):
        frames = oracle.sim_frames(cpu, c)
        oracle.sim_advance(cpu, c, seed, 0, k, oracle.plan(frames, threads=4))
    dist = np.hypot(gpu.ego_x - cpu.ego_x, gpu.ego_y - cpu.ego_y)
    same_lane = gpu.target_lane == cpu.target_lane
    print(f"free-running {ticks} ticks x {n} rollouts: max |d ego| {dist.max():.3e} m, "
          f"{(dist < 1e-6).mean():.3f} within 1e-6 m, target lane equal {same_lane.mean():.3f}")
    # trajectories differ by ~1e-13 (libdevice vs glibc transcendentals); a discrete decision can
    # flip on such a difference only at an exact threshold, so nearly every rollout stays together
    assert (dist < 1e-6).mean() >= 0.97


def test_simulator_model_on_cpu(pp, oracle):
    """The model with the oracle planner in the loop: cars keep their lanes' geometry, the ego
    accelerates from rest towards the speed limit and never leaves the road."""
    n, c, seed, k = 24, 12, 11, 1
    st = pp.RolloutStateHost(n, c)
    tbl = oracle.map_table()
    rng = np.random.default_rng(3)
    w = rng.integers(1, oracle.n_wp, n)
    st.ego_x[:] = tbl[w, 4]
    st.ego_y[:] = tbl[w, 5]
    st.ego_yaw_deg[:] = np.degrees(np.arctan2(tbl[w, 5] - tbl[w - 1, 5], tbl[w, 4] - tbl[w - 1, 4]))
    st.target_lane[:] = 1
    st.car_lane[:] = rng.integers(0, 3, (n, c))
    st.car_wp[:] = (w[:, None] + rng.integers(1, 4, (n, c))) % oracle.n_wp
    st.car_ratio[:] = rng.random((n, c))
    st.car_speed[:] = 17.88 + 8.94 * rng.random((n, c))
    speeds = []
    for _ in range(400):
        frames = oracle.sim_frames(st, c)
        assert np.isfinite(frames.car_x).all() and np.isfinite(frames.car_vx).all()
        v = np.hypot(frames.car_vx, frames.car_vy)
        assert np.allclose(v, st.car_speed, rtol=1e-12)
        plans = oracle.plan(frames, threads=4)
        assert (plans.n_points == 50).all()
        oracle.sim_advance(st, c, seed, 0, k, plans)
        assert ((st.car_ratio >= 0) & (st.car_ratio < 1.0 + 1e-12)).all()
        speeds.append(st.ego_speed_mph.copy())
    speeds = np.array(speeds)
    assert speeds[-1].max() <= 50.0 and np.median(speeds[-1]) > 25.0
    assert (np.abs(plans.ego_d - 6.0) < 7.0).all()
    assert st.tick == 400
