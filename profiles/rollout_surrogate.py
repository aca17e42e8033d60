"""Near misses of closed-loop rollouts: time to collision and time headway (include/pp.h,
pp_rollouts_set_surrogate).

    python profiles/rollout_surrogate.py [--rollouts 65536] [--ticks 3000] [--cars 12]
                                         [--cfg stock|fast_lane_change] [--traffic constant|idm]
    python profiles/rollout_surrogate.py --cost [--ticks 1000] [--rounds 2] ...

R rollouts x T ticks (consume_k = 1) with the near-miss measures on.  Prints one JSON line with
the card's name and power limit: ego-frames/s of the timed run; for front TTC, rear TTC and time
headway the exposure (seconds spent below 1 s and below 1.5 s per hour of driving, an hour of
driving being 180,000 ticks of 0.02 s), the share of rollouts whose minimum lies below 1 s, the
summed time histogram (0.02 s units) and the rollouts per bin of their minima; and, for the
rollouts with an incident (collision_rear excluded, as in the monitor), whether their worst front
TTC came before, at or after their first incident's tick.
--cost times the same job with the measures off and on (lean plans, no recorder), alternated
`rounds` times in one process after a warm-up of each, and prints the rates and their ratio.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rollout_incidents import card  # noqa: E402


def timed_run(pp, torch, args, cfg, ssm):
    ro = pp.Rollouts(pp.Map(), args.rollouts, args.cars, seed=args.seed, lean=True)
    ro.set_traffic(args.traffic)
    ro.set_surrogate(ssm)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    ro.run(args.ticks, 1, cfg=cfg)
    ev1.record()
    torch.cuda.synchronize()
    return ro, args.rollouts * args.ticks / (ev0.elapsed_time(ev1) * 1e-3)


def cost(pp, torch, args, cfg, base):
    def once(ssm):
        ro, _ = timed_run(pp, torch, argparse.Namespace(**{**vars(args), "ticks": 10}), cfg, ssm)
        del ro  # warm-up of this setting: scratch, module load
        ro, rate = timed_run(pp, torch, args, cfg, ssm)
        del ro
        torch.cuda.empty_cache()
        return rate

    once(False), once(True)
    rates = {"off": [], "on": []}
    for _ in range(args.rounds):
        rates["off"].append(once(False))
        rates["on"].append(once(True))
    off, on = (sum(rates[k]) / len(rates[k]) for k in ("off", "on"))
    return {**base, "metric": "closed-loop near-miss measures cost", "ego_frames_per_s": rates,
            "relative_to_off": on / off}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rollouts", type=int, default=65536)
    ap.add_argument("--ticks", type=int, default=None, help="default 3000, 1000 with --cost")
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
    abi = pp.abi
    cfg = pp.default_config()
    if args.cfg == "fast_lane_change":
        cfg.test_fast_lane_change = 1
    name, power = card()
    base = {"cfg": args.cfg, "traffic": args.traffic,
            "config": f"{args.rollouts} rollouts x {args.ticks} ticks, {args.cars} cars, consume_k=1, "
                      f"seed {args.seed}",
            "gpu": name or torch.cuda.get_device_name(0), "power_limit": power}
    if args.cost:
        print(json.dumps(cost(pp, torch, args, cfg, base)))
        return

    ro, rate = timed_run(pp, torch, args, cfg, True)
    tot = ro.surrogate_totals().cpu().numpy()
    rec = ro.surrogate()
    inc = ro.incidents()
    nb, mb = abi.SSM_BINS, abi.SSM_TOTAL_MIN
    hours = args.rollouts * args.ticks * 0.02 / 3600.0
    edges = abi.SSM_EDGES
    measures = {}
    for m, key in enumerate(abi.SSM_NAMES):
        hist = tot[m * nb:(m + 1) * nb]
        mins = tot[mb + m * nb:mb + (m + 1) * nb]
        measures[key] = {
            "exposure_s_per_hour_below_1s": float(hist[:edges.index(1.0) + 1].sum()) * 0.02 / hours,
            "exposure_s_per_hour_below_1.5s": float(hist[:edges.index(1.5) + 1].sum()) * 0.02 / hours,
            "rollouts_min_below_1s": float(mins[:edges.index(1.0) + 1].sum()) / args.rollouts,
            "rollouts_defined": int(np.isfinite(rec["min_" + key]).sum()),
            "time_hist": hist.tolist(), "min_hist": mins.tolist(),
        }
    first, worst = inc["first_tick"], rec["min_ttc_front_tick"]
    had = first >= 0
    order = {"rollouts_with_incident": int(had.sum()),
             "worst_ttc_front_before_first_tick": int((had & (worst >= 0) & (worst < first)).sum()),
             "worst_ttc_front_at_first_tick": int((had & (worst == first)).sum()),
             "worst_ttc_front_after_first_tick": int((had & (worst > first)).sum()),
             "no_ttc_front": int((had & (worst < 0)).sum())}
    kinds = inc["first_kind"]
    order["before_by_first_kind"] = {
        k: [int((had & (kinds == i)).sum()), int((had & (kinds == i) & (worst >= 0) & (worst < first)).sum())]
        for i, k in enumerate(abi.INC_NAMES) if (had & (kinds == i)).any()}
    line = {**base, "metric": "closed-loop near misses", "ego_frames_per_s": rate,
            "hours_driven": hours, "bin_edges_s": edges, "measures": measures, "incidents": order,
            "incident_counts": inc["count"].sum(axis=0).tolist(),
            "rollouts_nonfinite_distance": int((~np.isfinite(inc["distance_m"])).sum())}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
