"""The IDM traffic model of the rollouts on the GPU (include/pp.h, PP_TRAFFIC_IDM).

Tick by tick, under IDM: the frame the device built equals the CPU model's (bit-exact), the plan
for it equals the CPU planner's (teacher-forced), and the next state and the traffic record equal
the CPU restatement in traffic_oracle.c fed with the device's plans (bit-exact); the incident
record equals the monitor's restatement.  The result does not depend on stream groups, graph
replay, lean plans, how the ticks are split into runs or how the rollouts are sharded; selecting
the constant model changes nothing; and through the real planner the traffic stays within the
model's bounds.
"""
import os

import numpy as np
import pytest

import checkers
import incident_oracle
import traffic_oracle
from test_rollouts import STATE_FIELDS, assert_plans_match, cpu_state_from

abi = checkers.abi
INC = abi.INC


def assert_dicts_equal(got, want, where):
    for k in want:
        assert np.array_equal(got[k], want[k]), (where, k)


@pytest.mark.gpu
@pytest.mark.parametrize("n,c,ticks", [(192, 12, 40), (100, 64, 20)])
@pytest.mark.parametrize("consume_k", [1, 3])
def test_idm_ticks_match_cpu_model(pp, oracle, n, c, ticks, consume_k):
    seed, first = 77, 1000
    ro = pp.Rollouts(pp.Map(), n, c, seed=seed, first=first)
    ro.set_traffic("idm")
    prev = ro.state()
    tor = traffic_oracle.TrafficOracle()
    ts = tor.init(prev)
    assert_dicts_equal(ro.traffic(), ts.arrays, "initial")
    mon = incident_oracle.IncidentOracle()
    ms = mon.init(prev.ego_x, prev.ego_y)
    braking = 0
    for t in range(ticks):
        ro.run(1, consume_k)
        frames, plans = ro.last()
        now = ro.state()
        want_frames = oracle.sim_frames(prev, c)
        for k, a in frames.arrays().items():
            assert np.array_equal(a, getattr(want_frames, k)), (t, k)
        assert_plans_match(plans, oracle.plan(frames, threads=8), t)
        cpu = cpu_state_from(pp, prev)
        tor.advance(cpu, ts, seed, first, consume_k, plans)
        for k in STATE_FIELDS:
            assert np.array_equal(getattr(now, k), getattr(cpu, k)), (t, k)
        assert now.tick == cpu.tick == t + 1
        assert_dicts_equal(ro.traffic(), ts.arrays, t)
        mon.step(ms, c, consume_k, frames, plans, prev, now)
        assert_dicts_equal(ro.incidents(), ms.rec, t)
        braking += int((ts["car_acc"] < 0).sum())
        prev = now
    assert braking > 0  # cars did follow someone


def _job(pp, n, traffic="idm", groups=None, lean=False, graph=False, runs=(12,), k=2, first=0,
         seed=21):
    ro = pp.Rollouts(pp.Map(), n, 12, seed=seed, first=first, lean=lean)
    if traffic is not None:
        ro.set_traffic(traffic)
    if groups is not None:
        ro.set_groups(groups)
    if graph:
        os.environ["PP_ROLLOUT_GRAPH"] = "1"
    try:
        for t in runs:
            ro.run(t, k)
    finally:
        os.environ.pop("PP_ROLLOUT_GRAPH", None)
    st = ro.state()
    out = {f: getattr(st, f) for f in STATE_FIELDS}
    if traffic == "idm":
        out.update({"traffic." + k: v for k, v in ro.traffic().items()})
    out.update({"incidents." + k: v for k, v in ro.incidents().items()})
    return out, ro.stats().cpu().numpy()


@pytest.mark.gpu
def test_idm_does_not_depend_on_groups_graph_lean_or_run_split(pp):
    n, ticks = 12288, 40
    ref, ref_stats = _job(pp, n, groups=1, runs=(ticks,))
    variants = {
        "3 groups, graph replay": _job(pp, n, groups=3, graph=True, runs=(ticks,)),
        "lean": _job(pp, n, groups=1, lean=True, runs=(ticks,)),
        "T x run(1)": _job(pp, n, groups=1, runs=(1,) * ticks),
    }
    for name, (rec, stats) in variants.items():
        assert_dicts_equal(rec, ref, name)
        assert np.array_equal(stats, ref_stats), name
    assert (ref["traffic.car_acc"] < 0).any()


@pytest.mark.gpu
def test_idm_sharding(pp):
    n, ticks = 3000, 30
    whole, _ = _job(pp, 2 * n, runs=(ticks,))
    lo, _ = _job(pp, n, runs=(ticks,))
    hi, _ = _job(pp, n, runs=(ticks,), first=n)
    for k in whole:
        assert np.array_equal(whole[k], np.concatenate([lo[k], hi[k]])), k


@pytest.mark.gpu
def test_constant_model_is_the_default(pp):
    n, ticks = 6000, 30
    a, sa = _job(pp, n, traffic=None, runs=(ticks,))
    b, sb = _job(pp, n, traffic="constant", runs=(ticks,))
    assert_dicts_equal(b, a, "set_traffic(constant)")
    assert np.array_equal(sa, sb)
    ro = pp.Rollouts(pp.Map(), 64, 12)
    with pytest.raises(pp.PPError):
        ro.traffic()  # constant model: no IDM state
    with pytest.raises(pp.PPError):
        ro.set_traffic(7)
    ro.set_traffic("idm")
    ro.set_traffic("idm")  # again before the first tick: allowed
    ro.run(1, 1)
    with pytest.raises(pp.PPError):
        ro.set_traffic("constant")
    with pytest.raises(pp.PPError):
        ro.set_traffic("idm")
    assert ro.traffic()["car_v0"].shape == (64, 12)


def _planner_job(pp, traffic):
    ro = pp.Rollouts(pp.Map(), 4096, 12, seed=31, lean=True)
    ro.set_traffic(traffic)
    ro.run(1500, 1)
    return ro


@pytest.mark.gpu
def test_idm_through_the_planner(pp):
    const = _planner_job(pp, "constant")
    idm = _planner_job(pp, "idm")
    tr, st = idm.traffic(), idm.state()
    assert (tr["car_acc"] >= -abi.TRF_MAX_DEC).all() and (tr["car_acc"] <= abi.TRF_ACC).all()
    assert (st.car_speed >= 0).all() and (st.car_speed <= tr["car_v0"]).all()
    assert (tr["car_acc"] < 0).any()
    rear = {}
    for name, ro in (("constant", const), ("idm", idm)):
        stats = ro.stats().cpu().numpy()
        flags = {f: int(stats[abi.STAT_FLAG0 + i]) for i, f in enumerate(abi.FLAG_NAMES)}
        rec = ro.incidents()
        rear[name] = int(rec["count"][:, INC["collision_rear"]].sum())
        print(f"{name}: flags {flags}, incidents per kind {rec['count'].sum(axis=0).tolist()}")
    assert rear["idm"] < rear["constant"], rear
