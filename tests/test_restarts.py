"""The episode restarts of the rollouts on the GPU (include/pp.h, pp_rollouts_set_restart).

Episode 0 is pp_rollouts_create's draw; tick by tick, the device state, incident record, IDM state
and restart record equal the CPU restatement in restart_oracle.c fed with the device's own frames
and plans, bit for bit, including a non-finite restart of a long IDM run; the record does not
depend on stream groups, graph replay, lean plans, how the ticks are split into runs or how the
rollouts are sharded; the totals are the column sums and add up over shards; and a recorder with
the same mask freezes exactly where episode 1 begins.
"""
import os
import subprocess

import numpy as np
import pytest

import checkers
import restart_oracle
from test_rollouts import STATE_FIELDS, cpu_state_from

abi = checkers.abi
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL_BUT_REAR = [k for k in abi.INC_NAMES if k != "collision_rear"]
MASK = ALL_BUT_REAR + ["nonfinite"]


def limit_breaking_config(pp):
    """A planner that accelerates far beyond the monitor's limits, so that over-acceleration and
    over-speed restarts come within the first ticks."""
    cfg = pp.default_config()
    cfg.relaxed_acc, cfg.maximum_acc, cfg.max_speed = 30.0, 30.0, 40.0
    return cfg


def assert_dicts_equal(got, want, where):
    for k in want:
        assert np.array_equal(got[k], want[k], equal_nan=True), (where, k)


@pytest.fixture(scope="module")
def rso():
    return restart_oracle.RestartOracle()


@pytest.mark.gpu
@pytest.mark.parametrize("c", [12, 64])
def test_episode_0_is_the_create_draw(pp, rso, c):
    n, seed, first = 500, 77, 1000
    st = pp.Rollouts(pp.Map(), n, c, seed=seed, first=first).state()
    want = rso.draw(pp, seed, first, n, c)
    for k in STATE_FIELDS:
        assert np.array_equal(getattr(st, k), getattr(want, k)), k


def _check_ticks(pp, oracle, rso, ro, n, c, seed, first, consume_k, ticks, traffic, cfg, mask):
    """Run `ro` tick by tick against the restatement; returns the restart record."""
    prev = ro.state()
    ms = rso.monitor.init(prev.ego_x, prev.ego_y)
    ts = rso.traffic.init(prev) if traffic == "idm" else None
    rs = rso.init(n)
    for t in range(ticks):
        ro.run(1, consume_k, cfg=cfg)
        frames, plans = ro.last()
        now = ro.state()
        cpu = cpu_state_from(pp, prev)
        if ts is None:
            oracle.sim_advance(cpu, c, seed, first, consume_k, plans)
        else:
            rso.traffic.advance(cpu, ts, seed, first, consume_k, plans)
        rso.monitor.step(ms, c, consume_k, frames, plans, prev, cpu)
        rso.step(rs, cpu, ms, ts, c, seed, first, mask)
        for k in STATE_FIELDS:  # a plan may hold NaN points before the distance turns non-finite
            assert np.array_equal(getattr(now, k), getattr(cpu, k), equal_nan=True), (t, k)
        assert now.tick == cpu.tick == t + 1
        assert_dicts_equal(ro.incidents(), ms.rec, t)
        if ts is not None:
            assert_dicts_equal(ro.traffic(), ts.arrays, t)
        assert_dicts_equal(ro.restarts(), rs.rec, t)
        prev = now
    return rs.rec


@pytest.mark.gpu
@pytest.mark.parametrize("traffic", ["constant", "idm"])
@pytest.mark.parametrize("n,c", [(192, 12), (100, 64)])
@pytest.mark.parametrize("consume_k", [1, 3])
def test_restarts_match_cpu_tick_by_tick(pp, oracle, rso, traffic, n, c, consume_k):
    seed, first = 77, 1000
    ro = pp.Rollouts(pp.Map(), n, c, seed=seed, first=first)
    ro.set_restart(MASK)
    ro.set_traffic(traffic)
    rec = _check_ticks(pp, oracle, rso, ro, n, c, seed, first, consume_k, 90 // consume_k, traffic,
                       limit_breaking_config(pp), MASK)
    assert rec["episodes"].sum() > 0 and (rec["episodes"] >= 2).any()


# Rollout 169 of the 64-car IDM job with seed 2026 and consume_k 1 is the first whose distance
# turns non-finite, after tick 110 (tests/test_recorder.py); a job that starts at it reproduces it.
NONFINITE_ROLLOUT, NONFINITE_TICK = 169, 110


@pytest.mark.gpu
def test_nonfinite_restart_matches_cpu(pp, oracle, rso):
    n, c, seed = 8, 64, 2026
    ro = pp.Rollouts(pp.Map(), n, c, seed=seed, first=NONFINITE_ROLLOUT, lean=True)
    ro.set_traffic("idm")
    ro.set_restart(["nonfinite"])
    rec = _check_ticks(pp, oracle, rso, ro, n, c, seed, NONFINITE_ROLLOUT, 1, NONFINITE_TICK + 1,
                       "idm", None, ["nonfinite"])
    assert rec["by_bit"][0, abi.REC_NONFINITE] == 1
    assert rec["episode_tick"][0] == NONFINITE_TICK + 1
    assert np.isfinite(ro.incidents()["distance_m"]).all()


@pytest.mark.gpu
def test_long_idm_run_keeps_every_distance_finite(pp):
    # non-finite alone: with off_road in the mask most of these rollouts would restart at the
    # off-road incident that comes a few ticks before their distance turns non-finite
    ro = pp.Rollouts(pp.Map(), 8192, 64, seed=2026, lean=True)
    ro.set_traffic("idm")
    ro.set_restart(["nonfinite"])
    ro.run(1000, 1)
    rec, inc = ro.restarts(), ro.incidents()
    assert rec["by_bit"][:, abi.REC_NONFINITE].sum() == rec["episodes"].sum() > 0
    assert np.isfinite(inc["distance_m"]).all() and np.isfinite(rec["ended_m"]).all()
    assert (rec["ended_m"] <= inc["distance_m"]).all()
    print("restarts per ending bit:", dict(zip(abi.REC_NAMES, rec["by_bit"].sum(axis=0).tolist())))


def _job(pp, n=32768, groups=None, lean=False, graph=False, runs=(40,), first=0, traffic="idm"):
    ro = pp.Rollouts(pp.Map(), n, 12, seed=23, first=first, lean=lean)
    ro.set_traffic(traffic)
    ro.set_restart(MASK)
    if groups is not None:
        ro.set_groups(groups)
    if graph:
        os.environ["PP_ROLLOUT_GRAPH"] = "1"
    try:
        for t in runs:
            ro.run(t, 2, cfg=limit_breaking_config(pp))
    finally:
        os.environ.pop("PP_ROLLOUT_GRAPH", None)
    st = ro.state()
    out = {f: getattr(st, f) for f in STATE_FIELDS}
    out.update({"incidents." + k: v for k, v in ro.incidents().items()})
    out.update({"restarts." + k: v for k, v in ro.restarts().items()})
    out["totals"] = ro.restart_totals().cpu().numpy()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("traffic", ["constant", "idm"])
def test_restarts_do_not_depend_on_groups_graph_lean_or_run_split(pp, traffic):
    ref = _job(pp, groups=1, runs=(40,), traffic=traffic)
    assert ref["restarts.episodes"].sum() > 0
    variants = {
        "4 groups": _job(pp, groups=4, traffic=traffic),
        "8 groups, graph replay": _job(pp, groups=8, graph=True, traffic=traffic),
        "lean": _job(pp, groups=1, lean=True, traffic=traffic),
        "runs of 1, 9, 30": _job(pp, runs=(1, 9, 30), traffic=traffic),
        "40 runs of 1": _job(pp, runs=(1,) * 40, traffic=traffic),
    }
    for name, got in variants.items():
        for k in ref:
            assert np.array_equal(got[k], ref[k], equal_nan=True), (name, k)


@pytest.mark.gpu
def test_totals_are_the_column_sums_and_add_over_shards(pp):
    n = 16384
    whole = _job(pp, n, runs=(60,))
    tot = whole["totals"]
    assert tot.dtype == np.int64 and tot.shape == (abi.RST_TOTALS_LEN,)
    assert np.array_equal(tot[:abi.RST_BITS], whole["restarts.by_bit"].sum(axis=0))
    assert tot[abi.RST_TOTAL_LAPS] == whole["restarts.ended_lap"].sum()
    mm = whole["restarts.ended_m"] * 1000.0  # >= 0; llround rounds halves away from zero
    assert tot[abi.RST_TOTAL_MM] == np.floor(mm + 0.5).astype(np.int64).sum()
    assert tot[:abi.RST_BITS].sum() == whole["restarts.episodes"].sum() > 0
    lo = _job(pp, n // 2, runs=(60,))
    hi = _job(pp, n // 2, runs=(60,), first=n // 2)
    assert np.array_equal(lo["totals"] + hi["totals"], tot)
    for k in whole:
        if k != "totals":
            assert np.array_equal(np.concatenate([lo[k], hi[k]]), whole[k], equal_nan=True), k


@pytest.mark.gpu
def test_recorder_freezes_where_episode_1_begins(pp):
    ro = pp.Rollouts(pp.Map(), 4096, 12, seed=5, lean=True)
    ro.set_recorder(2, MASK)
    ro.set_restart(MASK)
    ro.run(120, 1, cfg=limit_breaking_config(pp))
    trig, rec = ro.recorder_triggers(), ro.restarts()
    frozen = trig["trigger_tick"] >= 0
    assert np.array_equal(frozen, rec["episodes"] >= 1) and frozen.any()
    if (rec["episodes"] == 1).any():
        one = rec["episodes"] == 1
        assert np.array_equal(trig["trigger_tick"][one] + 1, rec["episode_tick"][one])
    # the lowest fired bit of the frozen tick is the ending bit of episode 0 when it is the only one
    one = rec["episodes"] == 1
    low = np.array([(b & -b).bit_length() - 1 for b in trig["trigger_bits"][one].tolist()], dtype=np.int64)
    assert np.array_equal(rec["by_bit"][one][np.arange(one.sum()), low], np.ones(one.sum(), np.int64))


@pytest.mark.gpu
def test_restart_errors_and_off(pp):
    ro = pp.Rollouts(pp.Map(), 64, 12)
    for call in (ro.restarts, ro.restart_totals):
        with pytest.raises(pp.PPError):
            call()  # off
    with pytest.raises(pp.PPError):
        ro.set_restart(1 << (abi.REC_NONFINITE + 1))
    with pytest.raises(ValueError):
        ro.set_restart(["no_such_kind"])
    ro.set_restart(MASK)
    ro.set_restart(0)  # off again, before the first tick: allowed
    with pytest.raises(pp.PPError):
        ro.restarts()
    ro.set_restart(["nonfinite"])
    ro.run(1, 1)
    with pytest.raises(pp.PPError):
        ro.set_restart(MASK)
    assert ro.restarts()["by_bit"].shape == (64, abi.RST_BITS)


@pytest.mark.gpu
def test_a_rollout_that_never_restarts_is_unchanged(pp):
    """Every output of a rollout that never restarted equals the restart-off job's."""
    def job(mask):
        ro = pp.Rollouts(pp.Map(), 4096, 12, seed=19)
        ro.set_traffic("idm")
        if mask:
            ro.set_restart(mask)
        ro.run(100, 2)
        st = ro.state()
        out = {f: getattr(st, f) for f in STATE_FIELDS}
        out.update({"incidents." + k: v for k, v in ro.incidents().items()})
        out.update({"traffic." + k: v for k, v in ro.traffic().items()})
        _, pb = ro.last()
        out.update({"plans." + k: v for k, v in pb.arrays().items()})
        return out, (ro.restarts() if mask else None)
    off, _ = job(None)
    on, rec = job(MASK)
    kept = rec["episodes"] == 0
    assert kept.sum() > len(kept) // 2 and (~kept).any()
    for k in off:
        assert np.array_equal(on[k][kept], off[k][kept], equal_nan=True), k


@pytest.mark.gpu
def test_facade_restarts_equal_the_binding(pp, tmp_path):
    exe, out = str(tmp_path / "test_restarts"), str(tmp_path / "rst.bin")
    pkg = os.path.join(ROOT, "carnd-path-planning-project_b200")
    cmd = ["g++", "-std=c++11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_restarts.cpp"), "-L", pkg, "-lpp_b200",
           "-Wl,-rpath," + pkg, "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe, os.path.join(ROOT, "data", "highway_map.csv"), out],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "restarts facade ok" in res.stdout, (res.stdout, res.stderr)
    ro = pp.Rollouts(pp.Map(), 300, 12, seed=11, first=5)
    ro.set_restart(MASK)
    ro.set_traffic("idm")
    ro.run(40, 1)
    ro.run(20, 3)
    want = ro.restarts()
    order = [(name, want[name]) for name, _, _ in abi.RST_FIELDS]
    order.append(("totals", ro.restart_totals().cpu().numpy()))
    raw = open(out, "rb").read()
    pos = 0
    for name, a in order:
        got = np.frombuffer(raw, dtype=a.dtype, count=a.size, offset=pos).reshape(a.shape)
        pos += a.nbytes
        assert np.array_equal(got, a), name
    assert pos == len(raw)
