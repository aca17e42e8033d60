"""Episode restarts of closed-loop rollouts (include/pp.h, pp_rollouts_set_restart).

    python profiles/rollout_restarts.py [--rollouts 65536] [--ticks 3000] [--cars 12]
                                        [--cfg stock|fast_lane_change] [--traffic constant|idm]
    python profiles/rollout_restarts.py --cost [--ticks 1000] [--rounds 2] ...

Findings: R rollouts x T ticks (consume_k = 1, lean plans) restarting on every incident kind but
collision_rear and on a non-finite distance, timed against the same job with restarts off, in one
process.  Prints one JSON line with the card's name and power limit: ego-frames/s of both runs;
episodes per rollout; restarts per ending bit; the share of ended episodes that reached 4.32 miles
(the Udacity rubric); incidents per 100 miles over all driven distance (distance_m of every
rollout, which with restarts on is all the driving of the run); and the non-finite distances left
at the end of both runs.
--cost times the job with restarts off and with a rarely firing mask (front collisions only),
alternated `rounds` times after a warm-up of each, and prints the rates and their ratio.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rollout_incidents import METRES_PER_MILE, card  # noqa: E402

FINDINGS_MASK = [k for k in ("collision_front", "over_speed", "over_acc", "over_jerk", "out_of_lane",
                             "off_road")] + ["nonfinite"]


def timed_run(pp, torch, args, cfg, mask):
    ro = pp.Rollouts(pp.Map(), args.rollouts, args.cars, seed=args.seed, lean=True)
    ro.set_traffic(args.traffic)
    if mask:
        ro.set_restart(mask)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    ro.run(args.ticks, 1, cfg=cfg)
    ev1.record()
    torch.cuda.synchronize()
    return ro, args.rollouts * args.ticks / (ev0.elapsed_time(ev1) * 1e-3)


def cost(pp, torch, args, cfg, base):
    def once(mask):
        ro, _ = timed_run(pp, torch, argparse.Namespace(**{**vars(args), "ticks": 10}), cfg, mask)
        del ro  # warm-up of this setting: scratch, module load
        ro, rate = timed_run(pp, torch, args, cfg, mask)
        episodes = int(ro.restarts()["episodes"].sum()) if mask else 0
        del ro
        torch.cuda.empty_cache()
        return rate, episodes

    once(None), once(["collision_front"])
    rates, restarts = {"off": [], "on": []}, []
    for _ in range(args.rounds):
        rates["off"].append(once(None)[0])
        rate, ep = once(["collision_front"])
        rates["on"].append(rate)
        restarts.append(ep)
    off, on = (sum(rates[k]) / len(rates[k]) for k in ("off", "on"))
    return {**base, "metric": "closed-loop episode restarts cost", "mask": ["collision_front"],
            "ego_frames_per_s": rates, "restarts": restarts, "relative_to_off": on / off}


def findings(pp, torch, args, cfg, base):
    ro_off, rate_off = timed_run(pp, torch, args, cfg, None)
    nonfinite_off = int((~np.isfinite(ro_off.incidents()["distance_m"])).sum())
    del ro_off
    torch.cuda.empty_cache()
    ro, rate = timed_run(pp, torch, args, cfg, FINDINGS_MASK)
    rec, inc = ro.restarts(), ro.incidents()
    tot = ro.incident_totals().cpu().numpy()
    rtot = ro.restart_totals().cpu().numpy()
    ended = int(rec["episodes"].sum())
    miles = tot[pp.abi.INC_TOTAL_MM] / 1000.0 / METRES_PER_MILE
    return {
        **base, "metric": "closed-loop episode restarts", "mask": FINDINGS_MASK,
        "ego_frames_per_s": {"off": rate_off, "on": rate, "relative_to_off": rate / rate_off},
        "episodes_per_rollout": {"mean": float((rec["episodes"] + 1).mean()),
                                 "max": int(rec["episodes"].max() + 1)},
        "restarts_by_ending": {k: int(rtot[i]) for i, k in enumerate(pp.abi.REC_NAMES)},
        "ended_episodes": ended,
        "ended_lap_share": float(rtot[pp.abi.RST_TOTAL_LAPS]) / ended if ended else None,
        "miles": miles,
        "incidents_per_100_miles": {k: float(tot[i]) * 100.0 / miles
                                    for i, k in enumerate(pp.abi.INC_NAMES)},
        "nonfinite_distance_at_end": {"off": nonfinite_off,
                                      "on": int((~np.isfinite(inc["distance_m"])).sum())},
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rollouts", type=int, default=65536)
    ap.add_argument("--ticks", type=int, default=None)
    ap.add_argument("--cars", type=int, default=12)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--cfg", choices=["stock", "fast_lane_change"], default="stock")
    ap.add_argument("--traffic", choices=["constant", "idm"], default="constant")
    ap.add_argument("--cost", action="store_true")
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    if args.ticks is None:
        args.ticks = 1000 if args.cost else 3000

    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from __graft_entry__ import load_package
    pp = load_package()
    cfg = pp.default_config()
    if args.cfg == "fast_lane_change":
        cfg.test_fast_lane_change = 1
    name, power = card()
    base = {"cfg": args.cfg, "traffic": args.traffic,
            "config": f"{args.rollouts} rollouts x {args.ticks} ticks, {args.cars} cars, "
                      f"consume_k=1, seed {args.seed}",
            "gpu": name or torch.cuda.get_device_name(0), "power_limit": power}
    line = cost(pp, torch, args, cfg, base) if args.cost else findings(pp, torch, args, cfg, base)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
