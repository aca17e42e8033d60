"""The near-miss measures of the rollouts on the GPU (include/pp.h, pp_rollouts_set_surrogate).

Tick by tick, the device record equals the CPU restatement in surrogate_oracle.c fed with the
device's own frames, plans and car states, bit for bit, under both traffic models; the observer
changes nothing else the rollouts compute; the record does not depend on stream groups, graph
replay, lean plans or how the ticks are split into runs; the totals are the column sums and add
up over shards; and through the real planner the measures are defined and finite.
"""
import os
import subprocess

import numpy as np
import pytest

import checkers
import surrogate_oracle
from test_rollouts import STATE_FIELDS

abi = checkers.abi
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL_BUT_REAR = [k for k in abi.INC_NAMES if k != "collision_rear"]
MINS = ["min_ttc_front", "min_ttc_rear", "min_thw"]


def assert_records_equal(got, want, where):
    for k in want:
        assert np.array_equal(got[k], want[k]), (where, k)


@pytest.mark.gpu
@pytest.mark.parametrize("traffic", ["constant", "idm"])
@pytest.mark.parametrize("n,c", [(192, 12), (100, 64)])
@pytest.mark.parametrize("consume_k", [1, 3])
def test_surrogate_matches_cpu_tick_by_tick(pp, traffic, n, c, consume_k):
    # 9 s of driving: the egos start at rest, and only once they are up to speed do they close
    # on the cars ahead, so that every measure is defined somewhere
    ticks = 450 // consume_k
    ro = pp.Rollouts(pp.Map(), n, c, seed=77, first=1000)
    ro.set_traffic(traffic)
    ro.set_surrogate()
    so = surrogate_oracle.SurrogateOracle()
    ss = so.init(n)
    assert_records_equal(ro.surrogate(), ss.rec, "initial")
    for t in range(ticks):
        ro.run(1, consume_k)
        frames, plans = ro.last()
        so.step(ss, c, consume_k, frames, plans, ro.state())
        assert_records_equal(ro.surrogate(), ss.rec, t)
    rec = ss.rec
    for k in MINS:
        assert np.isfinite(rec[k]).any(), k
    assert rec["time_hist"].sum() > 0


def _observed_job(pp, traffic, ssm, n=4096, ticks=200):
    ro = pp.Rollouts(pp.Map(), n, 12, seed=19)
    ro.set_traffic(traffic)
    ro.set_recorder(5, ALL_BUT_REAR + ["nonfinite"])
    if ssm:
        ro.set_surrogate()
    ro.run(ticks // 2, 2)
    ro.run(ticks - ticks // 2, 1)
    st = ro.state()
    out = {f: getattr(st, f) for f in STATE_FIELDS}
    out.update({"incidents." + key: v for key, v in ro.incidents().items()})
    out["incident_totals"] = ro.incident_totals().cpu().numpy()
    if traffic == "idm":
        out.update({"traffic." + key: v for key, v in ro.traffic().items()})
    fb, pb = ro.last()
    out.update({"frames." + key: v for key, v in fb.arrays().items()})
    out.update({"plans." + key: v for key, v in pb.arrays().items()})
    out["stats"] = ro.stats().cpu().numpy()
    rec = ro.recording()
    out.update({"recording." + key: rec[key] for key in ("trigger_tick", "trigger_bits", "tick")})
    out.update({"recording.frames." + key: v for key, v in rec["frames"].arrays().items()})
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("traffic", ["constant", "idm"])
def test_surrogate_is_an_observer(pp, traffic):
    off, on = _observed_job(pp, traffic, False), _observed_job(pp, traffic, True)
    assert (off["recording.trigger_tick"] >= 0).any()
    for key in off:
        assert np.array_equal(on[key], off[key], equal_nan=True), key


def _job(pp, n=8192, groups=None, lean=False, graph=False, runs=(40,), first=0, traffic="idm"):
    ro = pp.Rollouts(pp.Map(), n, 12, seed=23, first=first, lean=lean)
    ro.set_traffic(traffic)
    ro.set_surrogate()
    if groups is not None:
        ro.set_groups(groups)
    if graph:
        os.environ["PP_ROLLOUT_GRAPH"] = "1"
    try:
        for t in runs:
            ro.run(t, 2)
    finally:
        os.environ.pop("PP_ROLLOUT_GRAPH", None)
    return ro.surrogate(), ro.surrogate_totals().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("traffic", ["constant", "idm"])
def test_surrogate_does_not_depend_on_groups_graph_lean_or_run_split(pp, traffic):
    ref, ref_tot = _job(pp, groups=1, runs=(40,), traffic=traffic)
    variants = {
        "3 groups, graph replay": _job(pp, groups=3, graph=True, runs=(40,), traffic=traffic),
        "lean": _job(pp, groups=1, lean=True, runs=(40,), traffic=traffic),
        "runs of 1, 9, 30": _job(pp, runs=(1, 9, 30), traffic=traffic),
    }
    for name, (rec, tot) in variants.items():
        assert_records_equal(rec, ref, name)
        assert np.array_equal(tot, ref_tot), name
    assert np.isfinite(ref["min_thw"]).any()


@pytest.mark.gpu
def test_surrogate_totals_are_the_column_sums_and_add_over_shards(pp):
    n = 6000
    rec, tot = _job(pp, n, runs=(300,))
    assert tot.dtype == np.int64 and tot.shape == (abi.SSM_TOTALS_LEN,)
    mb = abi.SSM_MEASURES * abi.SSM_BINS
    assert np.array_equal(tot[:mb], rec["time_hist"].sum(axis=0).reshape(-1))
    edges = np.array(abi.SSM_EDGES)
    for m, key in enumerate(MINS):
        b = (rec[key][:, None] >= edges[None, :]).sum(axis=1)  # comparisons only, as defined
        want = np.bincount(b, minlength=abi.SSM_BINS + 1)[:abi.SSM_BINS]
        assert np.array_equal(tot[abi.SSM_TOTAL_MIN + m * abi.SSM_BINS:][:abi.SSM_BINS], want), key
    assert tot[:mb].sum() > 0 and tot[mb:].sum() > 0
    lo, lo_tot = _job(pp, n // 2, runs=(300,))
    hi, hi_tot = _job(pp, n // 2, runs=(300,), first=n // 2)
    assert np.array_equal(lo_tot + hi_tot, tot)
    for k in rec:
        assert np.array_equal(np.concatenate([lo[k], hi[k]]), rec[k]), k


@pytest.mark.gpu
def test_surrogate_errors(pp):
    ro = pp.Rollouts(pp.Map(), 64, 12)
    with pytest.raises(pp.PPError):
        ro.surrogate()  # off
    with pytest.raises(pp.PPError):
        ro.surrogate_totals()
    ro.set_surrogate()
    ro.set_surrogate(False)  # off again, before the first tick: allowed
    with pytest.raises(pp.PPError):
        ro.surrogate()
    ro.set_surrogate()
    ro.run(1, 1)
    for on in (True, False):
        with pytest.raises(pp.PPError):
            ro.set_surrogate(on)
    assert ro.surrogate()["time_hist"].shape == (64, abi.SSM_MEASURES, abi.SSM_BINS)
    off = pp.Rollouts(pp.Map(), 64, 12)
    off.run(1, 1)
    with pytest.raises(pp.PPError):
        off.set_surrogate()


@pytest.mark.gpu
def test_surrogate_through_the_planner(pp):
    ro = pp.Rollouts(pp.Map(), 4096, 12, seed=31, lean=True)
    ro.set_traffic("idm")
    ro.set_surrogate()
    ro.run(1500, 1)
    rec = ro.surrogate()
    for k in MINS:
        v = rec[k]
        assert not np.isnan(v).any() and (v >= 0).all(), k
        share = np.isfinite(v).mean()
        assert share > 0, k
        print(f"{k}: finite in {share:.3f} of the rollouts, median {np.median(v[np.isfinite(v)]):.3f} s")
    front = np.isfinite(rec["min_ttc_front"])
    assert np.array_equal(front, rec["min_ttc_front_tick"] >= 0)
    assert ((rec["min_ttc_front_tick"] < 1500) & (rec["min_ttc_front_tick"] >= -1)).all()
    hist = rec["time_hist"].sum(axis=0)
    assert (hist.sum(axis=1) > 0).all()
    print("time_hist per measure (0.02 s units):", hist.tolist())


@pytest.mark.gpu
def test_facade_surrogate_equals_the_binding(pp, tmp_path):
    exe, out = str(tmp_path / "test_surrogate"), str(tmp_path / "ssm.bin")
    pkg = os.path.join(ROOT, "carnd-path-planning-project_b200")
    cmd = ["g++", "-std=c++11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_surrogate.cpp"), "-L", pkg, "-lpp_b200",
           "-Wl,-rpath," + pkg, "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe, os.path.join(ROOT, "data", "highway_map.csv"), out],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "surrogate facade ok" in res.stdout, (res.stdout, res.stderr)
    ro = pp.Rollouts(pp.Map(), 300, 12, seed=11, first=5)
    ro.set_traffic("idm")
    ro.set_surrogate()
    ro.run(40, 1)
    ro.run(20, 3)
    want = ro.surrogate()
    order = [(name, want[name]) for name, _, _ in abi.SSM_FIELDS]
    order.append(("totals", ro.surrogate_totals().cpu().numpy()))
    raw = open(out, "rb").read()
    pos = 0
    for name, a in order:
        got = np.frombuffer(raw, dtype=a.dtype, count=a.size, offset=pos).reshape(a.shape)
        pos += a.nbytes
        assert np.array_equal(got, a), name
    assert pos == len(raw)
