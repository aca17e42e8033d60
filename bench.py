#!/usr/bin/env python
"""bench.py — planned frames/sec at 1M-frame batches (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes, after the timed steps, what the last timed step computed (rank 0) as
DIR/<name>.npy in float64, at most 64 MB in all: per-frame (per-rollout) arrays at a fixed seeded
sample of the frames when all of them do not fit, DIR/sample_index.npy naming the frames.  The
inputs depend on the arguments alone, so two builds run with the same arguments can be compared
file for file.

Secondary lines (not the headline): --workload rollouts (BASELINE configs[2], closed-loop
ego-frames/s), --workload sweep (configs[3], candidate trajectories/s), --cars 64 (configs[4]).

Default run: N=1, 50 timed steps after 3 warm-ups (a few seconds).

One "step" = one pass of the hot path (pp_plan_batch, then the aggregate
statistics kernel; for N>1 followed by the NCCL all-reduce of the statistics
vector — the only collective on the path) over one batch of synthetic frames
that is already resident in HBM.  Workload at every N: BASELINE.json configs[1],
1,048,576 independent synthetic frames x 12 cars PER GPU (weak scaling; rank r
plans frames [r*2^20, (r+1)*2^20) of one global counter-based stream).

Prints ONE JSON line (rank 0).  `value` = frames of all ranks / max-over-ranks
device time; `e2e` = the same metric through pp_plan_batch_host with pinned HOST
buffers (H2D + D2H inside the timed region); `roofline` = algorithmic bytes
(1,520 B/frame, SURVEY §8d) / kernel time against the measured HBM peak, plus
the FP64-issue view that actually bounds this kernel (DESIGN.md §2);
`cpu_baseline` = the reference's own planner classes (oracle/_ref, kind
"reference") or the C restatement (kind "port") on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os

# before torch / CUDA start: the planner runs nine streams, the default is 8 hardware work
# queues (pp_api.cu, INTEGRATION.md "Threading")
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FRAMES_PER_GPU = 1 << 20
N_CARS = 12
SEED = 0x5EED
BYTES_IN = 204 + 36 * N_CARS   # SURVEY §8d
BYTES_OUT = 884
WORKLOAD = "configs[1]: 1,048,576 independent synthetic frames x 12 cars x 3 lanes per GPU"
METRIC = "planned frames/sec at 1M-frame batch"


# Library chatter (e.g. "NCCL version ..." goes to fd 1) must not share stdout with the ONE JSON
# line: fd 1 is pointed at stderr for the whole run and the line is written to the saved fd.
_REAL_STDOUT = None


def quiet_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 64_000_000  # --dump-outputs: all files together
DUMP_SEED = 0xD1


def sample_outputs(rows, whole):
    """--dump-outputs: `rows` (torch tensors or numpy arrays with one row per frame / rollout)
    at every row, or at a fixed seeded sample of rows when they would not fit in DUMP_BYTES,
    and `whole` (small arrays) as they are.  Tensors are gathered on their device, so the
    result survives later work on the buffers and the copy to the host can wait
    (write_outputs)."""
    import numpy as np
    import torch
    n = len(next(iter(rows.values())))
    row_bytes = 8 * (1 + sum(int(np.prod(v.shape[1:])) for v in rows.values()))
    headers = 128 * (1 + len(rows) + len(whole))  # one .npy header per file
    fit = (DUMP_BYTES - headers - 8 * sum(int(np.prod(v.shape)) for v in whole.values())) // row_bytes
    idx = np.arange(n) if n <= fit else \
        np.sort(np.random.default_rng(DUMP_SEED).choice(n, fit, replace=False))
    out = {"sample_index": idx, **whole}
    for k, v in rows.items():
        out[k] = v[torch.from_numpy(idx).to(v.device)] if torch.is_tensor(v) else v[idx]
    return out


def write_outputs(out_dir, arrays):
    """Each array as out_dir/<name>.npy in float64 (the integers the path computes are below
    2**53, flags below 2**31)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        v = v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
        np.save(os.path.join(out_dir, k + ".npy"), v.astype(np.float64))


def dump_outputs(out_dir, rows, whole):
    write_outputs(out_dir, sample_outputs(rows, whole))


def cpu_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_checker():
    import checkers  # TEST INFRASTRUCTURE (oracle/): used only as the timed CPU baseline
    if checkers.available("ref"):
        return checkers.Checker("ref"), "reference"
    return checkers.Checker("oracle"), "port"


def time_cpu(pp, m, n_frames, passes=1, cars=N_CARS, bufs=None):
    """Reference CPU implementation of the path on all host threads.  bufs: (frames, plans) to
    reuse between calls."""
    chk, kind = cpu_checker()
    threads = cpu_threads()
    if bufs is None:
        bufs = (pp.synth_frames(m, n_frames, cars, seed=SEED),
                pp.PlanBatch(n_frames, max(cars, 1), diag=True, cars=False))
    frames, plans = bufs
    best = float("inf")
    for _ in range(passes):
        t0 = time.perf_counter()
        chk.plan_into(frames, plans, threads=threads, want_flags=False)
        best = min(best, time.perf_counter() - t0)
    return n_frames / best, best, kind, threads


def run_reference(args):
    """--impl reference: the reference's own CPU planner, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from __graft_entry__ import load_package
    pp = load_package()
    m = pp.Map()
    n = args.frames or FRAMES_PER_GPU  # the same frames per step as the repo arm
    bufs = (pp.synth_frames(m, n, args.cars, seed=SEED),
            pp.PlanBatch(n, max(args.cars, 1), diag=True, cars=False))
    total_t, total_f = 0.0, 0
    kind, threads = None, None
    for i in range(args.warmup + args.steps):
        fps, t, kind, threads = time_cpu(pp, m, n, cars=args.cars, bufs=bufs)
        if i >= args.warmup:
            total_t += t
            total_f += n
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, bufs[1].arrays(), {})
    value = total_f / total_t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_t / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD if n == FRAMES_PER_GPU and args.cars == N_CARS else
                   f"{n} independent synthetic frames x {args.cars} cars x 3 lanes",
                   "frames_per_gpu": n, "cars_per_frame": args.cars,
                   "sample": f"all {n} frames of the workload per step"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": kind,
                         "sample": f"{n} frames per step, {threads} threads, "
                                   f"{'reference classes (oracle/_ref)' if kind == 'reference' else 'C restatement'}"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


def fp64_roofline(kernel):
    """The compute-bound workloads' roofline: share of the FP64 pipe's cycles the dominant kernel
    keeps busy (ncu sm__pipe_fp64_cycles_active, committed capture profiles/fp64_view.json) — the
    FP64 (non-tensor) issue rate of the B200 measured with profiles/fp64_peak.cu is the peak."""
    try:
        v = json.load(open(os.path.join(ROOT, "profiles", "fp64_view.json")))
        k = v["kernels"][kernel]
        pct = k["fp64_pipe_active_pct"]
        return {"bound": "fp64", "kernel": kernel, "achieved": pct * v["fp64_peak"]["tflops"] / 100.0,
                "peak": v["fp64_peak"]["tflops"], "unit": "TFLOP/s-equivalent of FP64 pipe cycles",
                "frac": pct / 100.0, "issue_active_pct": k["issue_active_pct"],
                "active_lanes_per_warp_instr": k["active_lanes_per_warp_instr"],
                "traffic": None, "source": v["source"]}
    except Exception:
        return None


def run_rollouts(args):
    """BASELINE configs[2]: closed-loop rollouts, device-resident simulator + planner.
    One step = --ticks ticks of every rollout; value = ego-frames (rollout-ticks) per second."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from __graft_entry__ import load_package
    pp = load_package()
    m = pp.Map()
    n, ticks = args.rollouts, args.ticks
    ro = pp.Rollouts(m, n, args.cars, seed=SEED, first=rank * n, lean=True)
    ro.run(max(3, min(20, ticks)), args.consume_k)  # warm-up ticks (also leaves the cold start)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    # (a job of thousands of short launches: NVML polled every 2 ms from another thread costs it
    # 2 % and its steadiness, profiles/r2_rollouts_sampler.log; every 20 ms it does not)
    sampler = ClockSampler(local, period_s=0.02) if rank == 0 else None
    launches0 = pp.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = args.steps
    ev0.record()
    for _ in range(steps):
        ro.run(ticks, args.consume_k)
    st = ro.stats()
    if world > 1:
        dist.all_reduce(st)
    ev1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    if rank == 0:
        stats = st.cpu().numpy()
        if args.dump_outputs:
            state = ro.state()
            dump_outputs(args.dump_outputs,
                         {k: getattr(state, k) for k, _, _ in pp.abi.ROLLOUT_STATE_FIELDS},
                         {"stats": stats})
        line = {"metric": "closed-loop ego-frames/sec (rollout-ticks)",
                "value": world * n * ticks * steps / (ms * 1e-3), "unit": "frames/s",
                "n_gpus": world, "steps": steps, "warmup": 3, "ms_per_step": ms / steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": f"configs[2]: {n} closed-loop rollouts x {ticks} ticks per GPU, "
                                       f"{args.cars} cars, consume_k={args.consume_k}",
                           "ms_per_tick": ms / steps / ticks},
                "gpu_launches": int(pp.launch_count() - launches0), "clocks": clocks,
                "roofline": {"bound": "launch latency", "note": "a tick is a chain of eight dependent "
                             "short kernels per stream group (8 groups); the simulator kernels keep "
                             "the issue slots 3-5 % busy", "sim_kernels": {
                                 k: fp64_roofline(k) for k in ("k_sim_frames", "k_sim_advance")}},
                "stats": {"frames": int(stats[0]), "points": int(stats[1]),
                          "lane_changes": int(stats[8])}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_sweep(args):
    """BASELINE configs[3]: candidate sweep, 384 candidates per frame (compute bound).
    One step = pp_sweep_batch over --frames frames (default 32,768); value = candidates/s."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from __graft_entry__ import load_package
    pp = load_package()
    m = pp.Map()
    n = args.frames if args.frames != FRAMES_PER_GPU else 32768
    frames = pp.synth_frames(m, n, args.cars, seed=SEED, first_frame=rank * n)
    df = pp.DeviceFrames(frames)
    steps = args.steps
    for _ in range(max(3, args.warmup)):
        out = pp.sweep_batch(m, df, want_scores=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = pp.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        out = pp.sweep_batch(m, df, want_scores=False)
    ev1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {k: v for k, v in out.items() if v is not None}, {})
        cands = 384
        best = out["best"].cpu().numpy()
        line = {"metric": "sweep candidates/sec (384 candidate trajectories per frame)",
                "value": world * n * cands * steps / (ms * 1e-3), "unit": "candidates/s",
                "n_gpus": world, "steps": steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"configs[3]: {n} frames x 384 candidates (3 lanes x 16 speeds x "
                                       f"8 times) per GPU, {args.cars} cars",
                           "frames_per_s": world * n * steps / (ms * 1e-3)},
                "gpu_launches": int(pp.launch_count() - launches0), "clocks": clocks,
                "roofline": fp64_roofline("k_sweep_emit"),
                "stats": {"winning_lane_hist": [int((best // 128 == k).sum()) for k in range(3)]}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


class ClockSampler:
    """SM clock + throttle reasons sampled every ~2 ms through NVML on a thread while the
    timed region runs (nvidia-smi's own loop is too coarse for a sub-second region)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap"}

    def __init__(self, index, period_s=0.002):
        import threading
        self.period_s = float(os.environ.get("PP_BENCH_CLOCK_MS", period_s * 1e3)) * 1e-3
        self.samples, self.maxes, self.reasons = [], [], set()
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = None
            try:  # the CUDA ordinal need not be the NVML index (CUDA_VISIBLE_DEVICES)
                import torch
                uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.h = None
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            # first NVML queries can take > 100 ms (longer than the whole timed region): pay for
            # them here, not on the sampling thread
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons"):
                pynvml.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            else:
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.ok = True
        except Exception:
            self.ok = False
        self.t = threading.Thread(target=self._run, daemon=True)
        if self.ok:
            self.t.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) \
                    if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period_s)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.ok:
            return out
        self.stop_flag = True
        self.t.join(timeout=2)
        sm = sorted(self.samples)
        if sm:
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz,
                   "reasons": sorted(self.reasons), "samples": len(sm)}
        return out


def bind_to_gpu_numa(local):
    """Pin this rank's threads (and, by first touch, its pinned host buffers) to the CPUs of the
    NUMA node its GPU hangs off: with one process per GPU all ranks otherwise share node 0's
    cores and memory for their staging copies.  Returns what was done, for the record."""
    info = {"numa_node": None, "cpus": len(os.sched_getaffinity(0)), "bound": False}
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info.update(cpus=len(cpus), bound=True)
    except Exception as e:  # not fatal: the measurement runs unbound
        info["error"] = str(e)[:80]
    return info


def make_comm(pp, dist, rank, world):
    """An ncclComm_t made through the C ABI (pp_comm_*); torch.distributed only carries rank 0's
    128-byte id to the other ranks."""
    def exchange(raw):
        box = [raw if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]
    return pp.Comm(rank, world, exchange if world > 1 else None)


def single_rank_stats(pp, m, world, n, cars, first_of_rank, torch, df, dp):
    """The statistics of all ranks' shards planned on THIS device alone (the N-rank reduced
    vector must equal it bit for bit): shards generated in HBM one after the other, into the
    rank's own buffers (df / dp are overwritten; the last shard generated is rank 0's again)."""
    from carnd_path_planning_project_b200 import parallel
    tot_i = torch.zeros(pp.STATS_LEN, dtype=torch.int64, device="cuda")
    tot_f = None
    for r in list(range(1, world)) + [0]:
        pp.synth_frames_dev(m, n, cars, seed=SEED, first_frame=first_of_rank(r), out=df)
        st = pp.plan_stats_batch(m, df, dp)
        fs = pp.fstats_batch(dp)
        tot_i += st
        tot_f = fs.clone() if tot_f is None else parallel.merge_fstats(tot_f, fs, pp.FSTAT_NMIN)
    torch.cuda.synchronize()
    return tot_i, tot_f


def traffic_for(cars):
    """ncu dram__bytes_read+write of the pipeline's kernels, from the committed capture of THIS
    car count (profiles/traffic.json, profiles/traffic_c64.json); None when there is none."""
    name = "traffic.json" if cars == N_CARS else f"traffic_c{cars}.json"
    prof = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(prof):
        return None, {}, None, None
    try:
        tj = json.load(open(prof))
        if int(tj.get("cars_per_frame", N_CARS)) != cars:
            return None, {}, None, None
        by_kernel = tj.get("dram_bytes_per_launch", {})
        per_frame = sum(by_kernel.values()) / float(tj["frames_per_launch"])
        view = {k: tj.get(k) for k in ("fp64_pipe_active_pct", "issue_active_pct",
                                       "active_lanes_per_warp_instr")}
        return per_frame, by_kernel, view, tj.get("source")
    except Exception:
        return None, {}, None, None


def cpu_baseline_legs(pp, m, n, cars):
    """BASELINE.md §3: the reference's own classes on all host threads (the figure of record),
    on one thread, and once with the reference's own build flags (no -O) — the last two on
    bounded samples."""
    import checkers
    fps, secs, kind, threads = time_cpu(pp, m, n, cars=cars)
    out = {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind,
           "sample": f"{n} frames of the workload, 1 pass, {threads} threads ({secs:.1f} s wall)"}
    small = min(n, 1 << 16)
    frames = pp.synth_frames(m, small, cars, seed=SEED)
    plans = pp.PlanBatch(small, max(cars, 1), diag=True, cars=False)
    chk, _ = cpu_checker()
    t0 = time.perf_counter()
    chk.plan_into(frames, plans, threads=1, want_flags=False)
    out["one_thread"] = {"value": small / (time.perf_counter() - t0), "unit": "frames/s",
                         "cores": 1, "sample": f"first {small} frames, 1 thread, -O2"}
    if checkers.available("ref_O0"):
        slow = checkers.Checker("ref_O0")
        tiny = min(small, 1 << 14)
        fr = frames.slice(0, tiny)
        pl = pp.PlanBatch(tiny, max(cars, 1), diag=True, cars=False)
        t0 = time.perf_counter()
        slow.plan_into(fr, pl, threads=1, want_flags=False)
        out["reference_flags_no_O"] = {
            "value": tiny / (time.perf_counter() - t0), "unit": "frames/s", "cores": 1,
            "sample": f"first {tiny} frames, 1 thread, the reference's own flags (-std=c++11, no -O)"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 50; dense64 3, sweep 5, rollouts 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=None,
                    help="frames per GPU (weak scaling) / in total (strong scaling)")
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-check", action="store_true",
                    help="skip the N-rank == 1-rank statistics check (N > 1)")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--cars", type=int, default=N_CARS,
                    help="cars per frame (12 = configs[1], the headline; 64 = configs[4])")
    ap.add_argument("--workload", default="frames",
                    choices=["frames", "dense64", "rollouts", "sweep"],
                    help="frames = BASELINE configs[1] (the headline metric, default); dense64 = "
                         "configs[4], 64M frames x 64 cars in total, generated in HBM and sharded; "
                         "rollouts = configs[2]; sweep = configs[3] (secondary lines)")
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="weak: --frames per GPU (default for frames); strong: --frames in total, "
                         "split over the GPUs (default for dense64)")
    ap.add_argument("--rollouts", type=int, default=65536, help="rollouts per GPU")
    ap.add_argument("--ticks", type=int, default=1000)
    ap.add_argument("--consume-k", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:  # (the reference arm plans the frames workload whatever --workload says)
        args.steps = 50 if args.impl == "reference" else \
            {"dense64": 3, "sweep": 5, "rollouts": 1}.get(args.workload, 50)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    quiet_stdout()
    if args.workload in ("rollouts", "sweep") and args.frames is None:
        args.frames = FRAMES_PER_GPU
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "rollouts":
        return run_rollouts(args)
    if args.workload == "sweep":
        return run_sweep(args)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    binding = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from __graft_entry__ import load_package
    pp = load_package()
    pp.set_kernel_variant(args.variant)

    dense = args.workload == "dense64"
    cars = 64 if dense else args.cars
    scaling = args.scaling or ("strong" if dense else "weak")
    if dense:
        total = args.frames or (64 << 20)
        cap = 32 << 20  # frames x 64 cars one B200 holds with its plans (108 GB)
        if scaling == "strong":
            n = min(total // world, cap)
        else:
            n = min(total, cap)
        workload = (f"configs[4]: {total} frames x 64 cars in total, generated in HBM "
                    f"(pp_synth_frames_dev), {n} frames resident per GPU"
                    + (" (the largest single-GPU slice)" if n * world < total else ""))
    else:
        per = args.frames or FRAMES_PER_GPU
        n = per // world if scaling == "strong" else per
        total = n * world
        workload = (WORKLOAD if cars == N_CARS and n == FRAMES_PER_GPU else
                    f"{n} independent synthetic frames x {cars} cars x 3 lanes per GPU")
    first_of_rank = lambda r: r * n  # noqa: E731  contiguous shards of one global stream
    mc = max(cars, 1)

    m = pp.Map()
    if dense:
        frames = None
        df = pp.synth_frames_dev(m, n, cars, seed=SEED, first_frame=first_of_rank(rank))
    else:
        frames = pp.synth_frames(m, n, cars, seed=SEED, first_frame=first_of_rank(rank))
        df = pp.DeviceFrames(frames)
    dp = pp.DevicePlans(n, mc, diag=True, cars=False)
    stream = torch.cuda.current_stream()
    comm = make_comm(pp, dist, rank, world)
    st_buf = torch.empty(pp.STATS_LEN, dtype=torch.int64, device="cuda")
    fs_buf = torch.empty(pp.FSTATS_LEN, dtype=torch.float64, device="cuda")

    def step():
        # plan + aggregate statistics in one call (pp_plan_stats_batch == pp_plan_batch followed
        # by pp_stats_batch; a chunk's statistics overlap the planning of the other chunks)
        return pp.plan_stats_batch(m, df, dp, out=st_buf)

    def final_reduce():
        # the f64 minima / maxima of the last plans, then the ONE collective of the job
        pp.fstats_batch(dp, out=fs_buf)
        comm.stats_reduce(st_buf, fs_buf)

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    final_reduce()
    fence()

    sampler = ClockSampler(local) if rank == 0 else None
    k_start = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    k_stop = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = pp.launch_count()
    fence()
    ev0.record(stream)
    for i in range(args.steps):
        step()
    final_reduce()
    ev1.record(stream)
    fence()
    launches = pp.launch_count() - launches0
    stats = st_buf.cpu().numpy().copy()
    fstats = fs_buf.cpu().numpy().copy()
    dump = None
    if args.dump_outputs and rank == 0:  # gathered on the device before the loops below plan into dp again
        dump = sample_outputs(dp.t, {"stats": stats, "fstats": fstats})
    # pp_plan_batch alone (the pipeline without the statistics pass), for the roofline
    for i in range(args.steps):
        k_start[i].record(stream)
        pp.plan_batch(m, df, dp)
        k_stop[i].record(stream)
    fence()
    clocks = sampler.stop() if sampler else None  # (both loops above run the GPU flat out)
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    # Per-kernel breakdown: in the timed region four chunks are in flight at once, so a kernel's
    # own duration cannot be read there.  A few extra (untimed) steps run the same launches
    # strictly one after the other with CUDA events around each kernel.
    pp.set_pipes(1)
    pp.set_phase_timing(True)
    bd_steps = 1 if dense else 3
    for _ in range(bd_steps):
        pp.plan_batch(m, df, dp)
    phase_ms, phase_chunks = pp.get_phase_ms()
    pp.set_phase_timing(False)
    pp.set_pipes(0)
    phase_ms = [v / bd_steps for v in phase_ms]
    phase_chunks //= bd_steps
    total_ms = ev0.elapsed_time(ev1)
    kern_ms = sum(a.elapsed_time(b) for a, b in zip(k_start, k_stop)) / args.steps
    t = torch.tensor([total_ms, kern_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kern_ms = float(t[0]), float(t[1])
    value = world * n * args.steps / (total_ms * 1e-3)

    # ---- the N-rank reduced statistics against a single-rank pass over the same frames ----
    stats_check = None
    if world > 1 and not args.no_check:
        if rank == 0:
            one_i, one_f = single_rank_stats(pp, m, world, n, cars, first_of_rank, torch, df, dp)
            assert np.array_equal(one_i.cpu().numpy(), stats), \
                ("N-rank int64 statistics differ from the single-rank pass", stats, one_i)
            assert np.array_equal(one_f.cpu().numpy(), fstats), \
                ("N-rank f64 statistics differ from the single-rank pass", fstats, one_f)
            stats_check = f"{world}-rank pp_stats_reduce == 1-rank pass over the same {world * n} frames (int64 and f64 vectors, bit for bit)"
        dist.barrier()

    # ---- end to end through the host entry point (pinned host buffers) ----
    e2e_n = n if not dense else min(n, 1 << 20)
    if frames is None:
        frames = pp.synth_frames(m, e2e_n, cars, seed=SEED, first_frame=first_of_rank(rank))
    hf = pp.FrameBatch(e2e_n, mc)
    for k, v in frames.arrays().items():
        pinned = torch.from_numpy(v[:e2e_n]).pin_memory()
        setattr(hf, k, pinned.numpy())
        hf.__dict__.setdefault("_keep", []).append(pinned)
    # what a drop-in caller asks for: the trajectories and the per-frame integers (the eight
    # f64 diagnostics and the followed-car ids stay optional outputs and are not requested)
    hp = pp.PlanBatch(e2e_n, mc, diag=False, cars=False)
    for k in hp.fields:
        pinned = torch.from_numpy(getattr(hp, k)).pin_memory()
        setattr(hp, k, pinned.numpy())
        hp.__dict__.setdefault("_keep", []).append(pinned)
    def time_e2e(call, probe):
        """frames/s from the MEDIAN step (wall clock around the call; the box's host and PCIe
        root are shared with other tenants, and one step in ten now and then takes twice as
        long, profiles/r2_e2e_pin.log), max over ranks; the mean is reported next to it."""
        call()  # warm-up (allocates the staging buffers)
        fence()
        secs = []
        for _ in range(args.e2e_steps):
            t0 = time.perf_counter()
            call()
            _ = float(np.nansum(probe[:16]))  # the step's result is on the host
            secs.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        te = torch.tensor([float(np.median(secs)), float(np.mean(secs))], dtype=torch.float64,
                          device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return world * e2e_n / float(te[0]), world * e2e_n / float(te[1])

    whole_value, whole_mean = time_e2e(lambda: pp.plan_batch_host(m, hf, hp), hp.n_points)
    whole_d2h = hp.bytes_per_frame() * e2e_n
    # the same job without sending the caller's own points back (pp_plan_batch_host_split): a
    # frame's first 10 points are its previous points verbatim (src/main.cpp:578), so only the
    # 40 new ones come down, plus all 50 of the frames that kept nothing
    keep, tail_len = pp.PREV_KEEP, pp.PATH_LEN - pp.PREV_KEEP
    sp = pp.PlanBatch(e2e_n, mc, diag=False, cars=False)
    sp.fields = [f for f in sp.fields if f not in ("next_x", "next_y")]
    sp.next_x = sp.next_y = None
    for k in sp.fields:
        setattr(sp, k, getattr(hp, k))  # the same pinned arrays
    tails = [torch.empty((e2e_n, tail_len), dtype=torch.float64).pin_memory() for _ in range(2)]
    heads = [torch.from_numpy(np.array(getattr(hf, k))).pin_memory() for k in ("prev_x", "prev_y")]
    tx, ty = tails[0].numpy(), tails[1].numpy()
    hx, hy = heads[0].numpy(), heads[1].numpy()
    want_x, want_y = hp.next_x.copy(), hp.next_y.copy()  # whole rows of the call above
    e2e_value, e2e_mean = time_e2e(lambda: pp.plan_batch_host_split(m, hf, sp, hx, hy, tx, ty),
                                   sp.n_points)
    full = sp.n_points == pp.PATH_LEN
    assert np.array_equal(tx, want_x[:, keep:], equal_nan=True) and \
        np.array_equal(ty, want_y[:, keep:], equal_nan=True) and \
        np.array_equal(hx[full], want_x[full, :keep], equal_nan=True) and \
        np.array_equal(hy[full], want_y[full, :keep], equal_nan=True), \
        "split rows differ from the whole rows"
    n_cold = int((hf.prev_n < keep).sum())
    e2e_d2h = (sp.bytes_per_frame() + 2 * 8 * tail_len) * e2e_n + 2 * 8 * keep * n_cold

    if rank == 0:
        peak, peak_src = peaks()
        bytes_in = 204 + 36 * cars  # SURVEY §8d
        alg_bytes = (bytes_in + BYTES_OUT) * n
        achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
        per_frame_traffic, traffic_by_kernel, ncu_view, traffic_src = traffic_for(cars)
        traffic = per_frame_traffic * n if per_frame_traffic is not None else None
        names = ["k_prep", "k_cars" if args.variant != 3 else "k_cars_t",
                 "k_decide_t", "k_emit", "side-stream tail (k_fallback/k_slow join)"]
        pipe_ms = sum(phase_ms)
        kernels = [{"name": nm, "ms_per_step": ms, "share": ms / pipe_ms if pipe_ms else None,
                    "launches_per_step": phase_chunks if nm[0] == "k" else None}
                   for nm, ms in zip(names, phase_ms)]
        # the dominant kernel on its own: algorithmic bytes it must move per frame (DESIGN.md §4)
        own_bytes = {names[0]: 204.0, names[1]: 36.0 * cars, names[2]: 160.0 + 76.0,
                     names[3]: 640.0 + 8.0}
        dom = max(kernels[:4], key=lambda k: k["ms_per_step"])
        dom_launches = max(1, phase_chunks)
        dom_ms = dom["ms_per_step"] / dom_launches
        dom_bytes = own_bytes[dom["name"]] * n / dom_launches
        dominant = {"kernel": dom["name"], "ms_per_launch": dom_ms, "launches_per_step": dom_launches,
                    "algorithmic_bytes_per_frame": own_bytes[dom["name"]],
                    "algorithmic_bytes_per_launch": dom_bytes,
                    "achieved": dom_bytes / (dom_ms * 1e-3) / 1e9, "unit": "GB/s",
                    "frac": dom_bytes / (dom_ms * 1e-3) / 1e9 / peak,
                    "traffic": traffic_by_kernel.get(dom["name"])}
        line = {
            "metric": METRIC if not dense else "planned frames/sec, 64 cars per frame (BASELINE configs[4])",
            "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload,
                       "frames_per_gpu": n, "frames_total": n * world, "cars_per_frame": cars,
                       "l2_policy": f"inputs+outputs ({(204 + 36 * cars + 884) * n / 1e9:.1f} GB per step) are larger than the 126 MB L2",
                       "kernel_variant": args.variant,
                       "step": "pp_plan_stats_batch (= pp_plan_batch + pp_stats_batch); after the "
                               "last step pp_fstats_batch + pp_stats_reduce (the one NCCL "
                               f"collective, {world} rank{'s' if world > 1 else ''})"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "mean_value": e2e_mean,
                    "timing": f"median of {args.e2e_steps} steps, wall clock around the call, max over ranks (mean_value: their mean)",
                    "h2d_bytes_per_step": int(hf.bytes_per_frame() * e2e_n),
                    "d2h_bytes_per_step": int(e2e_d2h),
                    "frames_per_step": e2e_n,
                    "host_binding": binding,
                    "host_buffer_bytes_per_frame": int(sp.bytes_per_frame() + 2 * 8 * tail_len),
                    "api": "pp_plan_batch_host_split (pinned host buffers, chunked H2D/plan/D2H "
                           "pipeline; outputs: the 40 new points of every trajectory, all 50 of the "
                           f"{n_cold} frames without kept points, n_points, lanes, ref_wp, flags; the "
                           "10 kept points of a trajectory are the caller's own prev_x/prev_y rows "
                           "and are not sent back; checked here against the whole rows, bit for bit)",
                    "whole_rows": {"value": whole_value, "mean_value": whole_mean, "unit": "frames/s",
                                   "d2h_bytes_per_step": int(whole_d2h),
                                   "api": "pp_plan_batch_host (next_x/next_y[50] rows, the kept "
                                          "points included)"}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "kernel": "pp_plan_batch pipeline (k_prep + k_cars + k_decide_t + k_emit, "
                                   "chunks of 262,144 frames, four planned concurrently); "
                                   "dominant: " + dom["name"],
                         "kernel_ms": kern_ms, "kernels": kernels, "dominant_kernel": dominant,
                         "kernels_one_after_the_other_ms": pipe_ms, "ncu": ncu_view,
                         "algorithmic_bytes_per_frame": bytes_in + BYTES_OUT,
                         "algorithmic_bytes_per_step": alg_bytes,
                         "note": "FP64-issue / divergence bound, not HBM bound (DESIGN.md §2): "
                                 f"{bytes_in + BYTES_OUT:,} B against tens of thousands of instructions per frame, a third to a half of them FP64"},
            "clocks": clocks,
            "stats": {"frames": int(stats[0]), "points": int(stats[1]),
                      "lane_changes": int(stats[8]),
                      "f64": {nm: float(v) for nm, v in zip(pp.FSTAT_NAMES, fstats)},
                      "check": stats_check},
        }
        if not args.no_cpu and world == 1:
            line["cpu_baseline"] = cpu_baseline_legs(pp, m, min(n, FRAMES_PER_GPU), cars)
        emit(line)
    comm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
