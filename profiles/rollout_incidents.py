"""Incidents of closed-loop rollouts: which planner configuration drives further without one.

    python profiles/rollout_incidents.py [--rollouts 65536] [--ticks 3000] [--cars 12]
                                         [--cfg stock|fast_lane_change] [--traffic constant|idm]

R rollouts x T ticks (default 65,536 x 3,000 = 60 s of driving each, consume_k = 1) with the
incident monitor of include/pp.h; prints one JSON line: ego-frames/s of the timed run, miles
driven, incidents per kind per 100 miles, the share of incident-free rollouts (collision_rear
excluded, as in the monitor's definition) and best_clean_m in miles (min, median, p99, max),
the planner's flag counts (BRAKE, MAXBRAKE, ADJUST, KEEP, ... summed over every frame), with the
card's name and power limit.  --cfg fast_lane_change sets the planner's test_fast_lane_change = 1,
everything else stays at the stock tunables.  --traffic idm selects the car-following traffic
model (pp_rollouts_set_traffic, include/pp.h) instead of the constant-speed one.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
METRES_PER_MILE = 1609.344


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:  # the line still carries torch's device name
        return None, None


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rollouts", type=int, default=65536)
    ap.add_argument("--ticks", type=int, default=3000)
    ap.add_argument("--cars", type=int, default=12)
    ap.add_argument("--consume-k", type=int, default=1)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--cfg", choices=["stock", "fast_lane_change"], default="stock")
    ap.add_argument("--traffic", choices=["constant", "idm"], default="constant")
    args = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from __graft_entry__ import load_package
    pp = load_package()
    cfg = pp.default_config()
    if args.cfg == "fast_lane_change":
        cfg.test_fast_lane_change = 1
    ro = pp.Rollouts(pp.Map(), args.rollouts, args.cars, seed=args.seed, lean=True)
    ro.set_traffic(args.traffic)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    ro.run(args.ticks, args.consume_k, cfg=cfg)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    tot = ro.incident_totals().cpu().numpy()
    rec = ro.incidents()
    stats = ro.stats().cpu().numpy()
    miles = tot[pp.abi.INC_TOTAL_MM] / 1000.0 / METRES_PER_MILE
    best = rec["best_clean_m"] / METRES_PER_MILE
    name, power = card()
    line = {
        "metric": "closed-loop incidents", "cfg": args.cfg, "traffic": args.traffic,
        "config": f"{args.rollouts} rollouts x {args.ticks} ticks, {args.cars} cars, "
                  f"consume_k={args.consume_k}, seed {args.seed}",
        "gpu": name or torch.cuda.get_device_name(0), "power_limit": power,
        "ego_frames_per_s": args.rollouts * args.ticks / (ms * 1e-3),
        "miles": miles,
        "incidents_per_100_miles": {k: float(tot[i]) * 100.0 / miles
                                    for i, k in enumerate(pp.abi.INC_NAMES)},
        "incidents": {k: int(tot[i]) for i, k in enumerate(pp.abi.INC_NAMES)},
        "incident_free_share": 1.0 - float(tot[pp.abi.INC_TOTAL_ROLLOUTS]) / args.rollouts,
        # an ego whose position became NaN or infinite poisons the millimetre total (llround)
        "rollouts_nonfinite_distance": int((~np.isfinite(rec["distance_m"])).sum()),
        "best_clean_miles": {"min": float(best.min()), "median": float(np.median(best)),
                             "p99": float(np.percentile(best, 99)), "max": float(best.max())},
        "flags": {f: int(stats[pp.abi.STAT_FLAG0 + i]) for i, f in enumerate(pp.abi.FLAG_NAMES)},
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
