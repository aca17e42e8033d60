"""What the rollouts' planner was given before they failed: the flight recorder (include/pp.h,
pp_rollouts_set_recorder) on a full closed-loop job, and a replay of sampled windows.

    python profiles/rollout_recorder.py [--rollouts 65536] [--ticks 3000] [--cars 12]
        [--traffic constant|idm] [--consume-k 1] [--window 256] [--sample 512] [--fixture-out F]

The job of rollout_incidents.py runs twice: with the recorder's mask at every incident kind but
collision_rear (the monitor's own "first incident"), then at a non-finite distance_m alone.  The
job is deterministic, so both runs see the same rollouts.  One JSON line, with the card's name and
power limit:
  - triggered rollouts per trigger bit, cross-checked against the incident record (the first
    tick and kind of every rollout, and the count of non-finite distances);
  - for a seeded sample of each class, every window replanned on the device (loop closure, bit
    for bit: tests/recorder_replay.py) and by the CPU oracle (the share of windows where it agrees
    with the device), the planner's flags in the last 10 ticks, and for non-finite windows the
    first tick whose plan holds a non-finite point and whether that tick's frame was finite.
--fixture-out writes the first sampled non-finite window (frames, ticks, consume_k, device plans)
as an .npz for tests/golden/.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from rollout_incidents import card  # noqa: E402
import recorder_replay  # noqa: E402


def replay(pp, oracle, rec, w, threads):
    """Replan the windows of `rec` on the device and with the oracle; per-window findings."""
    fb = rec["frames"]
    m = len(rec["tick"])
    df, dp = pp.DeviceFrames(fb), pp.DevicePlans(fb.n, fb.max_cars, diag=False, cars=False)
    pp.plan_batch(pp.Map(), df, dp)
    dev = dp.to_host()
    ok, applies = recorder_replay.closure(fb, dev, rec["tick"], rec["consume_k"])
    # the oracle plans the filled frames that are all finite (a frame holding NaN is the
    # simulator's doing, not the planner's); the others count as agreeing
    filled = rec["tick"] >= 0
    finite = filled.reshape(-1) & recorder_replay.frame_finite(fb)
    rows = np.flatnonzero(finite)
    sub = pp.abi.FrameBatch(len(rows), fb.max_cars)
    for k in fb.arrays():
        setattr(sub, k, np.ascontiguousarray(getattr(fb, k)[rows]))
    t0 = time.time()
    part = oracle.plan(sub, threads=threads, diag=False, cars=False)
    cpu_s = time.time() - t0
    cpu = pp.abi.PlanBatch(fb.n, fb.max_cars, diag=False, cars=False)
    for k in cpu.fields:
        getattr(cpu, k)[...] = getattr(dev, k)
        getattr(cpu, k)[rows] = getattr(part, k)
    agree = recorder_replay.oracle_agrees(dev, cpu, m, w, finite.reshape(m, w))
    nfill = filled.sum(axis=1)
    flags = dev.flags.reshape(m, w)
    last10 = (np.arange(w)[None, :] >= (nfill - 10)[:, None]) & filled
    flag_counts = {name: int((((flags >> i) & 1).astype(bool) & last10).sum())
                   for i, name in enumerate(pp.abi.FLAG_NAMES)}
    flag_windows = {name: int(((((flags >> i) & 1).astype(bool) & last10).any(axis=1)).sum())
                    for i, name in enumerate(pp.abi.FLAG_NAMES)}
    out = {"windows": m, "frames": int(filled.sum()),
           "loop_closure_share": float(ok.sum() / max(applies.sum(), 1)),
           "oracle_agrees_share": float(agree.mean()) if m else None,
           "oracle_seconds": cpu_s,
           "flags_last10_frames": {k: v for k, v in flag_counts.items() if v},
           "flags_last10_windows": {k: v for k, v in flag_windows.items() if v}}
    return out, dev, cpu, ok, agree


def nonfinite_origin(fb, dev, cpu, tick, m, w, flag_names):
    """For each window: the first slot whose device plan holds a non-finite point, whether that
    slot's frame was all finite, and whether the oracle's plan of it is non-finite too."""
    npts = dev.n_points.reshape(m, w)
    nx, ny = dev.next_x.reshape(m, w, 50), dev.next_y.reshape(m, w, 50)
    inside = np.arange(50)[None, None, :] < npts[..., None]
    bad_plan = (~np.isfinite(nx) | ~np.isfinite(ny)) & inside
    bad_plan = bad_plan.any(axis=2) & (tick >= 0)
    cnx = cpu.next_x.reshape(m, w, 50)
    cpu_bad = ((~np.isfinite(cnx)) & (np.arange(50) < cpu.n_points.reshape(m, w)[..., None])).any(axis=2)
    fin = recorder_replay.frame_finite(fb).reshape(m, w)
    res = {"windows_with_a_nonfinite_plan": 0, "first_bad_plan_from_finite_frame": 0,
           "first_bad_plan_from_nonfinite_frame": 0, "oracle_also_nonfinite_there": 0,
           "flags_of_first_bad_plan": {}, "ticks_before_trigger": []}
    flags = dev.flags.reshape(m, w)
    last = (tick >= 0).sum(axis=1) - 1
    for i in range(m):
        js = np.flatnonzero(bad_plan[i])
        if not len(js):
            continue
        j = int(js[0])
        res["windows_with_a_nonfinite_plan"] += 1
        res["first_bad_plan_from_finite_frame" if fin[i, j] else "first_bad_plan_from_nonfinite_frame"] += 1
        res["oracle_also_nonfinite_there"] += int(cpu_bad[i, j])
        res["ticks_before_trigger"].append(int(last[i] - j))
        for b, name in enumerate(flag_names):
            if (int(flags[i, j]) >> b) & 1:
                res["flags_of_first_bad_plan"][name] = res["flags_of_first_bad_plan"].get(name, 0) + 1
    tb = res.pop("ticks_before_trigger")
    res["ticks_before_trigger"] = ({"min": int(min(tb)), "median": float(np.median(tb)), "max": int(max(tb))}
                                   if tb else None)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rollouts", type=int, default=65536)
    ap.add_argument("--ticks", type=int, default=3000)
    ap.add_argument("--cars", type=int, default=12)
    ap.add_argument("--consume-k", type=int, default=1)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--traffic", choices=["constant", "idm"], default="constant")
    ap.add_argument("--window", type=int, default=256)
    ap.add_argument("--sample", type=int, default=512)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
    ap.add_argument("--fixture-out", default=None)
    args = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from __graft_entry__ import load_package
    import checkers
    pp = load_package()
    oracle = checkers.Checker("oracle")
    names = pp.abi.REC_NAMES
    masks = {"first_incident": [k for k in pp.abi.INC_NAMES if k != "collision_rear"],
             "nonfinite": ["nonfinite"]}
    w = args.window
    name, power = card()
    line = {"metric": "closed-loop flight recorder", "traffic": args.traffic,
            "config": f"{args.rollouts} rollouts x {args.ticks} ticks, {args.cars} cars, "
                      f"consume_k={args.consume_k}, seed {args.seed}, window {w}, sample {args.sample}",
            "gpu": name or torch.cuda.get_device_name(0), "power_limit": power,
            "ring_bytes": args.rollouts * w * (200 + 32 * args.cars)}
    rng = np.random.default_rng(args.seed)
    for cls, mask in masks.items():
        ro = pp.Rollouts(pp.Map(), args.rollouts, args.cars, seed=args.seed, lean=True)
        ro.set_traffic(args.traffic)
        ro.set_recorder(w, mask)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        ro.run(args.ticks, args.consume_k)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        trig, inc = ro.recorder_triggers(), ro.incidents()
        frozen = trig["trigger_tick"] >= 0
        per_bit = {b: int(((trig["trigger_bits"] >> i) & 1).sum()) for i, b in enumerate(names)}
        res = {"ego_frames_per_s": args.rollouts * args.ticks / (ms * 1e-3),
               "triggered": int(frozen.sum()), "triggered_per_bit": {k: v for k, v in per_bit.items() if v}}
        if cls == "first_incident":
            lowest = np.where(frozen, np.log2((trig["trigger_bits"] & -trig["trigger_bits"].astype(np.int64))
                                              .clip(1)).astype(np.int64), -1)
            first_kinds = {k: int((inc["first_kind"] == i).sum()) for i, k in enumerate(pp.abi.INC_NAMES)}
            res["first_kind_counts_incidents"] = {k: v for k, v in first_kinds.items() if v}
            res["crosscheck_first_tick_equal"] = bool(np.array_equal(trig["trigger_tick"], inc["first_tick"]))
            res["crosscheck_first_kind_equal"] = bool(np.array_equal(lowest, inc["first_kind"]))
            first_rec = (inc["first_kind"].copy(), inc["first_tick"].copy())
        else:
            nonfinite = ~np.isfinite(inc["distance_m"])
            res["rollouts_nonfinite_distance"] = int(nonfinite.sum())
            res["crosscheck_nonfinite_equal"] = bool(np.array_equal(frozen, nonfinite))
            # the first incidents of the rollouts that end non-finite: which kind, and how many
            # ticks before the distance turns non-finite (0: the same tick)
            kind, ft = first_rec
            tt = trig["trigger_tick"]
            res["first_incident_of_nonfinite_rollouts"] = {
                k: {"rollouts": int(((kind == i) & nonfinite).sum()),
                    "same_tick": int(((kind == i) & nonfinite & (ft == tt)).sum()),
                    "1_to_10_ticks_before": int(((kind == i) & nonfinite & (tt - ft >= 1) & (tt - ft <= 10)).sum()),
                    "of_all_with_this_first_kind": int((kind == i).sum())}
                for i, k in enumerate(pp.abi.INC_NAMES) if (kind == i).any()}
            if frozen.any():
                i0 = int(np.flatnonzero(frozen)[np.argmin(trig["trigger_tick"][frozen])])
                res["earliest"] = {"rollout": i0, "trigger_tick": int(trig["trigger_tick"][i0])}
        pick = np.flatnonzero(frozen)
        if len(pick) > args.sample:
            pick = np.sort(rng.choice(pick, args.sample, replace=False))
        if len(pick):
            rec = ro.recording(pick)
            del ro
            torch.cuda.empty_cache()
            rep, dev, cpu, ok, agree = replay(pp, oracle, rec, w, args.threads)
            res["sample"] = rep
            if cls == "first_incident":
                kinds = {}
                for i, r in enumerate(pick):
                    kinds.setdefault(pp.abi.INC_NAMES[inc["first_kind"][r]], []).append(i)
                res["sample_by_first_kind"] = {}
                m = len(pick)
                flags = dev.flags.reshape(m, w)
                nfill = (rec["tick"] >= 0).sum(axis=1)
                speed = rec["frames"].ego_speed_mph.reshape(m, w)
                for kname, rows in kinds.items():
                    rows = np.array(rows)
                    last10 = np.arange(w)[None, :] >= (nfill[rows] - 10)[:, None]
                    fl = {f: int((((flags[rows] >> b) & 1).astype(bool) & last10).any(axis=1).sum())
                          for b, f in enumerate(pp.abi.FLAG_NAMES)}
                    res["sample_by_first_kind"][kname] = {
                        "windows": len(rows), "oracle_agrees": int(agree[rows].sum()),
                        "ego_mph_at_trigger_median": float(np.median(speed[rows, nfill[rows] - 1])),
                        "windows_with_flag_in_last10": {f: v for f, v in fl.items() if v}}
            else:
                res["nonfinite_origin"] = nonfinite_origin(rec["frames"], dev, cpu, rec["tick"], len(pick), w,
                                                          pp.abi.FLAG_NAMES)
                if args.fixture_out:
                    i = 0
                    rows = slice(i * w, (i + 1) * w)
                    fb = rec["frames"]
                    np.savez_compressed(
                        args.fixture_out, rollout=pick[i], seed=args.seed, cars=args.cars,
                        traffic=args.traffic, tick=rec["tick"][i], consume_k=rec["consume_k"][i],
                        trigger_tick=rec["trigger_tick"][i], trigger_bits=rec["trigger_bits"][i],
                        **{"in_" + k: getattr(fb, k)[rows] for k in fb.arrays()},
                        **{"dev_" + k: getattr(dev, k)[rows] for k in
                           ("next_x", "next_y", "n_points", "target_lane", "flags")})
        line[cls] = res
    print(json.dumps(line))


if __name__ == "__main__":
    main()
