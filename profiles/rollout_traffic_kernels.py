"""Device time per kernel and tick of the closed-loop rollouts under each traffic model.

    python profiles/rollout_traffic_kernels.py [--rollouts 65536] [--cars 12] [--ticks 200]

For each model (constant, idm): a fresh rollouts object (lean plans, the seed of
rollout_incidents.py), 300 ticks to get the traffic going, then --ticks ticks under torch.profiler
(CUDA activity only).  Prints one JSON line per model: microseconds of device time per tick for
every kernel, summed over its launches, with the card's name and power limit.  The planner's
kernels take different branches under different traffic, so their times move with the model too.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rollouts", type=int, default=65536)
    ap.add_argument("--cars", type=int, default=12)
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--seed", type=int, default=2026)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from __graft_entry__ import load_package
    from rollout_incidents import card
    assert torch.cuda.is_available(), "needs a CUDA device"
    pp = load_package()
    name, power = card()
    for model in ("constant", "idm"):
        ro = pp.Rollouts(pp.Map(), args.rollouts, args.cars, seed=args.seed, lean=True)
        ro.set_traffic(model)
        ro.run(300, 1)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ro.run(args.ticks, 1)
            torch.cuda.synchronize()
        per_tick = {}
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = e.self_cuda_time_total
            if t > 0:
                per_tick[e.key[:80]] = round(t / args.ticks, 2)
        per_tick = dict(sorted(per_tick.items(), key=lambda kv: -kv[1]))
        print(json.dumps({"metric": "device us per tick by kernel", "traffic": model,
                          "config": f"{args.rollouts} rollouts x {args.cars} cars, ticks "
                                    f"300-{300 + args.ticks}, consume_k=1, seed {args.seed}",
                          "gpu": name or torch.cuda.get_device_name(0), "power_limit": power,
                          "us_per_tick": per_tick}))
        ro.close()


if __name__ == "__main__":
    main()
