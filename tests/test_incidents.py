"""The incident monitor of the rollouts on the GPU (include/pp.h, pp_rollout_incidents).

Tick by tick, the device record equals the CPU restatement fed with the device's own frames,
plans and car states, every field bit for bit; the record does not depend on stream groups,
graph replay, lean plans or how the ticks are split into runs; the totals are the column sums;
and the incidents fire through the real planner when its tunables break the limits.  That the
monitor leaves the simulator itself unchanged is pinned by tests/test_rollouts.py, which checks
the state, frames, plans and statistics tick by tick against the CPU model.
"""
import os

import numpy as np
import pytest

import checkers
import incident_oracle

abi = checkers.abi
INC = abi.INC


def assert_records_equal(got, want, where):
    for k in want:
        assert np.array_equal(got[k], want[k]), (where, k, got[k][:4], want[k][:4])


@pytest.mark.gpu
@pytest.mark.parametrize("consume_k", [1, 3])
def test_incidents_match_cpu_monitor_tick_by_tick(pp, consume_k):
    n, c, seed, first, ticks = 192, 12, 77, 1000, 200
    m = pp.Map()
    ro = pp.Rollouts(m, n, c, seed=seed, first=first)
    prev = ro.state()
    mon = incident_oracle.IncidentOracle()
    ms = mon.init(prev.ego_x, prev.ego_y)
    assert_records_equal(ro.incidents(), ms.rec, "initial")
    for t in range(ticks):
        ro.run(1, consume_k)
        frames, plans = ro.last()
        now = ro.state()
        mon.step(ms, c, consume_k, frames, plans, prev, now)
        assert_records_equal(ro.incidents(), ms.rec, t)
        prev = now
    rec = ms.rec
    assert (rec["distance_m"] > 1.0).all() and (rec["max_speed"] > 1.0).all()
    print(f"k={consume_k}: incidents per kind {rec['count'].sum(axis=0).tolist()}, "
          f"rollouts with one {(rec['first_tick'] >= 0).sum()}")


def _job(pp, n, groups=None, lean=False, graph=False, runs=(12,), k=2):
    m = pp.Map()
    ro = pp.Rollouts(m, n, 12, seed=21, lean=lean)
    if groups is not None:
        ro.set_groups(groups)
    if graph:
        os.environ["PP_ROLLOUT_GRAPH"] = "1"
    try:
        for t in runs:
            ro.run(t, k)
    finally:
        os.environ.pop("PP_ROLLOUT_GRAPH", None)
    return ro.incidents(), ro.incident_totals().cpu().numpy(), ro.stats().cpu().numpy()


@pytest.mark.gpu
def test_incidents_do_not_depend_on_groups_graph_lean_or_run_split(pp):
    n, ticks = 12288, 40
    ref = _job(pp, n, groups=1, runs=(ticks,))
    variants = {
        "3 groups, graph replay": _job(pp, n, groups=3, graph=True, runs=(ticks,)),
        "lean": _job(pp, n, groups=1, lean=True, runs=(ticks,)),
        "T x run(1)": _job(pp, n, groups=1, runs=(1,) * ticks),
    }
    for name, (rec, tot, stats) in variants.items():
        assert_records_equal(rec, ref[0], name)
        assert np.array_equal(tot, ref[1]), name
        assert np.array_equal(stats, ref[2]), name
    assert ref[0]["distance_m"].min() > 0


@pytest.mark.gpu
def test_incident_totals_are_the_column_sums(pp):
    n = 6000
    ro = pp.Rollouts(pp.Map(), n, 12, seed=8)
    ro.run(300, 1)
    rec = ro.incidents()
    tot = ro.incident_totals().cpu().numpy()
    assert tot.dtype == np.int64 and tot.shape == (abi.INC_TOTALS_LEN,)
    assert np.array_equal(tot[:abi.INC_KINDS], rec["count"].sum(axis=0))
    assert tot[abi.INC_TOTAL_ROLLOUTS] == (rec["first_tick"] >= 0).sum()
    # llround: halves away from zero (distances are >= 0)
    assert tot[abi.INC_TOTAL_MM] == np.floor(rec["distance_m"] * 1000.0 + 0.5).astype(np.int64).sum()
    assert tot[abi.INC_TOTAL_MM] > 0


def _planner_job(pp, **tunables):
    cfg = pp.default_config()
    for k, v in tunables.items():
        setattr(cfg, k, v)
    ro = pp.Rollouts(pp.Map(), 4096, 12, seed=31, lean=True)
    ro.run(1500, 1, cfg=cfg)
    return ro.incidents()


@pytest.mark.gpu
def test_incidents_fire_through_the_planner(pp):
    stock = _planner_job(pp)
    fast = _planner_job(pp, max_speed=25.0)
    hard = _planner_job(pp, relaxed_acc=14.0, maximum_acc=14.0)
    sp = INC["over_speed"]
    assert stock["count"][:, sp].sum() == 0 and stock["max_speed"].max() <= 22.352
    # every rollout that reached speed logged it, and nearly all of them did
    reached = fast["max_speed"] > 22.352
    assert np.array_equal(reached, fast["count"][:, sp] > 0)
    assert reached.mean() > 0.9
    assert hard["count"][:, INC["over_acc"]].sum() > 0
    assert hard["max_acc"].max() > stock["max_acc"].max()
    for name, rec in (("stock", stock), ("max_speed 25", fast), ("acc 14", hard)):
        print(f"{name}: incidents per kind {rec['count'].sum(axis=0).tolist()}, "
              f"best clean median {np.median(rec['best_clean_m']):.0f} m")
