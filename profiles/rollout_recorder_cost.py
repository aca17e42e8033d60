"""What the flight recorder costs the closed-loop rollouts (include/pp.h, pp_rollouts_set_recorder).

    python profiles/rollout_recorder_cost.py [--rollouts 65536] [--ticks 1000] [--cars 12]
                                             [--traffic constant|idm] [--rounds 2]

R rollouts x T ticks with the recorder off, at W = 64 and at W = 256 (no trigger, so every
rollout stores every tick: the full cost), alternated `rounds` times in one process after a
warm-up of each.  Prints one JSON line: ego-frames/s of every run, the ring's bytes per setting,
with the card's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rollout_incidents import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rollouts", type=int, default=65536)
    ap.add_argument("--ticks", type=int, default=1000)
    ap.add_argument("--cars", type=int, default=12)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--traffic", choices=["constant", "idm"], default="constant")
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from __graft_entry__ import load_package
    pp = load_package()
    windows = [0, 64, 256]

    def run(w):
        ro = pp.Rollouts(pp.Map(), args.rollouts, args.cars, seed=args.seed, lean=True)
        ro.set_traffic(args.traffic)
        ro.set_recorder(w, 0)
        ro.run(10, 1)  # warm-up: scratch, module load
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        ro.run(args.ticks, 1)
        ev1.record()
        torch.cuda.synchronize()
        rate = args.rollouts * args.ticks / (ev0.elapsed_time(ev1) * 1e-3)
        del ro
        torch.cuda.empty_cache()
        return rate

    for w in windows:  # warm-up of every setting
        run(w)
    rates = {w: [] for w in windows}
    for _ in range(args.rounds):
        for w in windows:
            rates[w].append(run(w))
    name, power = card()
    off = sum(rates[0]) / len(rates[0])
    line = {"metric": "closed-loop flight recorder cost", "traffic": args.traffic,
            "config": f"{args.rollouts} rollouts x {args.ticks} ticks, {args.cars} cars, consume_k=1, "
                      f"seed {args.seed}, triggers 0",
            "gpu": name or torch.cuda.get_device_name(0), "power_limit": power,
            "ego_frames_per_s": {("off" if w == 0 else f"W={w}"): r for w, r in rates.items()},
            "relative_to_off": {f"W={w}": sum(rates[w]) / len(rates[w]) / off for w in windows if w},
            "ring_bytes": {f"W={w}": args.rollouts * w * (200 + 32 * args.cars) for w in windows if w}}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
