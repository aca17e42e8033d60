"""GPU parity beyond the defaults: planner tunables other than the reference's literals, and
cars held over from earlier messages (pp_frames::car_frozen_*), on every kernel variant and
through the host entry points, against the CPU oracle (oracle/pp_oracle.c).

Bars as everywhere: integers and + - * / sqrt quantities bit for bit, trajectories within
1e-9 relative and 1e-6 m.  The oracle's own use of each tunable and of the frozen fields is
pinned on the CPU (test_oracle_config_cpu.py).
"""
import numpy as np
import pytest

import checkers
from conftest import assert_plans_equal, plans_dict

pytestmark = pytest.mark.gpu

abi = checkers.abi
ALL_FLAGS = (1 << abi.NUM_FLAGS) - 1
VARIANTS = (1, 2, 3, 4, 0)  # fused, strided pipeline, tiled pipeline, warp per frame, auto
# flags each config is meant to drive (the matrix must actually reach those paths)
TARGETED = {"tight": ("ACC_OVERRIDE", "CURV_ADJUST", "KEEP", "ADJUST", "FALLBACK"),
            "loose": ("ACC_OVERRIDE", "ADJUST"), "max25": ("ACC_OVERRIDE",),
            "edges": ("BRAKE", "MAXBRAKE", "ADJUST")}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def gmap(pp, torch_cuda):
    return pp.Map()


def gpu_plan(pp, torch, m, fb, cfg=None, variant=0):
    df = pp.DeviceFrames(fb)
    dp = pp.DevicePlans(fb.n, fb.max_cars, diag=True, cars=True)
    pp.set_kernel_variant(variant)
    try:
        before = pp.launch_count()
        pp.plan_batch(m, df, dp, cfg=cfg)
        torch.cuda.synchronize()
        assert pp.launch_count() > before
    finally:
        pp.set_kernel_variant(0)
    return dp.to_host()


def live_slots(fb):
    return np.arange(fb.max_cars)[None, :] < np.minimum(fb.n_cars, fb.max_cars)[:, None]


def assert_matches(got, want, fb, what):
    """assert_plans_equal over the written car slots only (slots at and beyond n_cars are not
    written by the device)."""
    live = live_slots(fb)
    g, w = plans_dict(got), plans_dict(want)
    for k in abi.PLAN_CARS:
        g[k], w[k] = g[k][live], w[k][live]
    assert_plans_equal(g, w, ALL_FLAGS, bitwise_traj=False, what=what)


def flag_count(plans, name):
    return int(((plans.flags & abi.FLAG[name]) != 0).sum())


@pytest.mark.parametrize("cfg_name", list(checkers.CONFIGS))
@pytest.mark.parametrize("cars,n", [(12, 6000), (64, 1000)])
def test_config_matrix_on_every_variant(pp, torch_cuda, gmap, oracle, cfg_name, cars, n):
    """Each config on every kernel variant (auto takes the pipeline at 6,000 frames and the
    warp-per-frame kernel at 1,000) against oracle.plan(frames, cfg)."""
    cfg = checkers.config(cfg_name)
    fb = pp.synth_frames(gmap, n, cars, seed=500 + cars, rare_permille=100)
    want = oracle.plan(fb, threads=8, cfg=cfg)
    for v in VARIANTS:
        got = gpu_plan(pp, torch_cuda, gmap, fb, cfg, v)
        assert_matches(got, want, fb, f"{cfg_name} variant {v}: ")
    if cfg_name == "default":
        return
    base = oracle.plan(fb, threads=8)
    moved = (want.target_time != base.target_time) | (want.flags != base.flags) | \
        (want.target_lane != base.target_lane) | (want.ego_acc != base.ego_acc)
    assert moved.sum() > 0.02 * n, (cfg_name, int(moved.sum()))
    for name in TARGETED[cfg_name]:
        assert flag_count(want, name) > 0, (cfg_name, name)
    if cfg_name == "tight":
        assert flag_count(want, "CURV_ADJUST") > 2 * flag_count(base, "CURV_ADJUST")
        assert flag_count(want, "KEEP") > flag_count(base, "KEEP")
    elif cfg_name == "edges":
        assert flag_count(want, "KEEP") == 0 and flag_count(base, "KEEP") > 0
        assert flag_count(want, "BRAKE") > flag_count(base, "BRAKE")
    elif cfg_name == "max25":
        assert (want.target_speed == 25.0).any()
    elif cfg_name == "loose":
        assert flag_count(want, "ACC_OVERRIDE") > flag_count(base, "ACC_OVERRIDE")


def followed_frozen(fb, plans, pick):
    """Frames whose next_car_id or next_car_in_target_lane is a held-over car."""
    rows = np.arange(fb.n)
    hit = np.zeros(fb.n, bool)
    for k in ("next_car_id", "next_car_in_target_lane"):
        ids = getattr(plans, k)
        j = np.argmax(fb.car_id == ids[:, None], axis=1)
        hit |= (ids >= 0) & pick[rows, j] & (j < fb.n_cars)
    return hit


@pytest.mark.parametrize("cars,n,cfg_name", [(1, 5003, "default"), (5, 4999, "tight"),
                                             (12, 6001, "default"), (33, 4101, "edges"),
                                             (64, 4203, "tight")])
def test_held_over_cars_on_every_variant(pp, torch_cuda, gmap, oracle, cars, n, cfg_name):
    """~30 % of the matched slots held over with stale values (s +-30 m, d and lane moved, vs
    scaled) and their positions NaN, ragged n_cars: every variant and tile geometry against the
    oracle."""
    cfg = checkers.config(cfg_name)
    rng = np.random.default_rng(cars)
    fb = pp.synth_frames(gmap, n, cars, seed=600 + cars, rare_permille=100, max_cars=cars)
    if cars > 1:
        fb.n_cars[::3] = rng.integers(0, cars + 1, len(fb.n_cars[::3]))
    frozen, pick = checkers.hold_over(fb, oracle.plan(fb, threads=8, cfg=cfg), rng)
    assert pick.sum() > 0.15 * live_slots(fb).sum()
    want = oracle.plan(frozen, threads=8, cfg=cfg)
    assert (want.car_lane[pick] == frozen.car_frozen_lane[pick]).all()
    for v in VARIANTS:
        got = gpu_plan(pp, torch_cuda, gmap, frozen, cfg, v)
        assert_matches(got, want, frozen, f"held over, {cars} cars, variant {v}: ")
    assert followed_frozen(frozen, want, pick).sum() > 20  # LimitSpeed saw held-over cars


def test_held_over_cars_across_pipeline_chunks(pp, torch_cuda, gmap, oracle):
    """70,000 frames: three pipeline chunks, frozen slots in every one of them, so a wrong
    per-chunk offset of the frozen arrays shows."""
    n, cfg = 70000, checkers.config("tight")
    fb = pp.synth_frames(gmap, n, 12, seed=71, rare_permille=50)
    frozen, pick = checkers.hold_over(fb, oracle.plan(fb, threads=8, cfg=cfg),
                                      np.random.default_rng(71))
    for lo, hi in ((0, 32768), (32768, 65536), (65536, n)):
        assert pick[lo:hi].sum() > 0.2 * pick.sum() * (hi - lo) / n
    want = oracle.plan(frozen, threads=8, cfg=cfg)
    for v in (2, 3):
        got = gpu_plan(pp, torch_cuda, gmap, frozen, cfg, v)
        assert_matches(got, want, frozen, f"variant {v}: ")


@pytest.mark.parametrize("variant", [0, 4])
def test_cars_frozen_at_their_own_device_results(pp, torch_cuda, gmap, variant):
    """Freeze matched cars at the device's own matching results and hide their positions: every
    output stays bit-identical except car_next_wp of the frozen slots, which becomes 0."""
    cfg = checkers.config("tight")
    fb = pp.synth_frames(gmap, 6000, 12, seed=81, rare_permille=150)
    want = gpu_plan(pp, torch_cuda, gmap, fb, cfg, variant)
    frozen, pick = checkers.hold_over(fb, want, np.random.default_rng(81), stale=False)
    got = gpu_plan(pp, torch_cuda, gmap, frozen, cfg, variant)
    live = live_slots(fb)
    for k in got.fields:
        a, b = getattr(got, k), getattr(want, k)
        if k == "car_next_wp":
            assert (a[pick] == 0).all() and np.array_equal(a[live & ~pick], b[live & ~pick])
        elif k in abi.PLAN_CARS:
            assert np.array_equal(a[live], b[live], equal_nan=True), k
        else:
            assert np.array_equal(a, b, equal_nan=True), k


def test_host_entry_points_with_held_over_cars_and_a_config(pp, torch_cuda, gmap, oracle):
    """40,000 frames (more than the first host chunk of 32,768) with held-over cars and the
    tight config: pageable and page-locked buffers and the split-rows call, each bit for bit the
    device entry point, which matches the oracle."""
    n, cfg = 40000, checkers.config("tight")
    fb = pp.synth_frames(gmap, n, 12, seed=91, rare_permille=60)
    fb.prev_n[::9] = 0
    frozen, pick = checkers.hold_over(fb, oracle.plan(fb, threads=8, cfg=cfg),
                                      np.random.default_rng(91))
    assert pick[32768:].any()
    dev = gpu_plan(pp, torch_cuda, gmap, frozen, cfg)
    assert_matches(dev, oracle.plan(frozen, threads=8, cfg=cfg), frozen, "device: ")
    host = pp.plan_batch_host(gmap, frozen, cfg=cfg)
    for k in host.fields:
        assert np.array_equal(getattr(host, k), getattr(dev, k), equal_nan=True), ("pageable", k)
    pf = pp.FrameBatch(n, frozen.max_cars)
    for k in list(frozen.arrays()) + [name for name, _ in abi.FROZEN_FIELDS]:
        setattr(pf, k, pp.pinned_like(getattr(frozen, k)))
    got = pp.PlanBatch(n, frozen.max_cars)
    for k in got.fields:
        setattr(got, k, pp.pinned_like(getattr(got, k)))
    pp.plan_batch_host(gmap, pf, got, cfg=cfg)
    for k in got.fields:
        assert np.array_equal(getattr(got, k), getattr(dev, k), equal_nan=True), ("page-locked", k)
    keep, tail_len = abi.PREV_KEEP, abi.PATH_LEN - abi.PREV_KEEP
    sp = pp.PlanBatch(n, frozen.max_cars)
    sp.next_x = sp.next_y = None
    sp.fields = [f for f in sp.fields if f not in ("next_x", "next_y")]
    head_x, head_y = frozen.prev_x.copy(), frozen.prev_y.copy()
    tail_x, tail_y = np.full((n, tail_len), -1.0), np.full((n, tail_len), -1.0)
    pp.plan_batch_host_split(gmap, frozen, sp, head_x, head_y, tail_x, tail_y, cfg=cfg)
    for k in sp.fields:
        assert np.array_equal(getattr(sp, k), getattr(dev, k), equal_nan=True), ("split", k)
    whole = (dev.n_points == abi.PATH_LEN) | (frozen.prev_n < keep)
    assert whole.mean() > 0.9
    assert np.array_equal(np.concatenate([head_x, tail_x], axis=1)[whole], dev.next_x[whole], equal_nan=True)
    assert np.array_equal(np.concatenate([head_y, tail_y], axis=1)[whole], dev.next_y[whole], equal_nan=True)


# ---- unit entry points with other tunables ---------------------------------------------------

def dev_arr(T, a, dtype=None):
    return T.from_numpy(np.ascontiguousarray(a, dtype=dtype)).cuda()


def ptr(t):
    import ctypes as C
    return C.c_void_p(t.data_ptr())


@pytest.mark.parametrize("cfg_name", ["tight", "edges"])
def test_unit_entry_points_with_other_configs(pp, torch_cuda, gmap, oracle, golden_units, cfg_name):
    """pp_lane_change_batch, pp_limit_speed_batch and pp_trajectory_build_batch on the golden
    unit inputs against the oracle's _cfg units: bit for bit, points within the trajectory bars;
    and the config does move each of them."""
    import ctypes as C
    T, g, cfg = torch_cuda, golden_units, checkers.config(cfg_name)
    # lane change
    cs, cvs = g["lc_cars"]
    es, evs, dt0 = g["lc_ego"]
    n, nc = g["lc_id"].shape
    out = T.zeros(n, dtype=T.int32, device="cuda")
    args = [dev_arr(T, g["lc_id"], np.int32), dev_arr(T, cs), dev_arr(T, cvs),
            dev_arr(T, g["lc_lane"], np.int32)]
    sc = [dev_arr(T, g["lc_el"], np.int32), dev_arr(T, g["lc_tl"], np.int32), dev_arr(T, es),
          dev_arr(T, evs), dev_arr(T, dt0)]
    assert pp.lib.pp_lane_change_batch(C.byref(cfg), *[ptr(t) for t in args], nc,
                                       *[ptr(t) for t in sc], ptr(out), C.c_int64(n), None) == 0
    want = oracle.lane_change(g["lc_id"], cs, cvs, g["lc_lane"], g["lc_el"], g["lc_tl"], es, evs,
                              dt0, cfg=cfg)
    assert np.array_equal(out.cpu().numpy(), want)
    if cfg_name == "tight":
        assert (want != g["lc_out"]).any()
    # limit speed + speed controller
    ins = [dev_arr(T, a) for a in g["ls_in"]]
    inl = dev_arr(T, g["ls_inlane"], np.int32)
    m = inl.numel()
    outs = [T.zeros(m, dtype=T.float64, device="cuda") for _ in range(4)]
    fl = T.zeros(m, dtype=T.int32, device="cuda")
    assert pp.lib.pp_limit_speed_batch(C.byref(cfg), *[ptr(t) for t in ins], ptr(inl),
                                       *[ptr(t) for t in outs], ptr(fl), C.c_int64(m), None) == 0
    want = oracle.limit_speed(*g["ls_in"], g["ls_inlane"], cfg=cfg)
    for o, k in zip(outs, ("ls_speed", "ls_time", "sc_speed", "sc_time")):
        assert np.array_equal(o.cpu().numpy(), want[k]), k
        assert (want[k] != g["ls_" + k]).any(), k
    assert np.array_equal(fl.cpu().numpy().view(np.uint32), want["flags"])
    # trajectory builder (maximum_acc)
    ex, ey, yaw, ed, evd, start, target, time = g["tr_ego"]
    k = len(ex)
    ox, oy = (T.zeros((k, 50), dtype=T.float64, device="cuda") for _ in range(2))
    on, tf = (T.zeros(k, dtype=T.int32, device="cuda") for _ in range(2))
    a = [dev_arr(T, g["tr_prev_n"], np.int32), dev_arr(T, g["tr_prev_x"]), dev_arr(T, g["tr_prev_y"]),
         dev_arr(T, ex), dev_arr(T, ey), dev_arr(T, yaw), dev_arr(T, g["tr_tl"], np.int32),
         dev_arr(T, ed), dev_arr(T, evd), dev_arr(T, start), dev_arr(T, target), dev_arr(T, time)]
    assert pp.lib.pp_trajectory_build_batch(gmap.handle, C.byref(cfg), *[ptr(t) for t in a],
                                            ptr(ox), ptr(oy), ptr(on), ptr(tf), C.c_int64(k),
                                            None) == 0
    wx, wy, wn, wf = oracle.trajectory_build(g["tr_prev_n"], g["tr_prev_x"], g["tr_prev_y"], ex, ey,
                                             yaw, g["tr_tl"], ed, evd, start, target, time, cfg=cfg)
    assert np.array_equal(on.cpu().numpy(), wn)
    mask = sum(abi.FLAG[f] for f in ("ACC_OVERRIDE", "CURV_ADJUST", "ACCT_HIGH", "ACCN_HIGH",
                                     "FALLBACK", "SPLINE_INPUT_ERR"))
    assert np.array_equal(tf.cpu().numpy().view(np.uint32) & mask, wf & mask)
    for got, want_xy in ((ox.cpu().numpy(), wx), (oy.cpu().numpy(), wy)):
        assert np.array_equal(got != got, want_xy != want_xy)
        assert np.nanmax(np.abs(got - want_xy)) <= 1e-6
        assert np.nanmax(np.abs(got - want_xy) / np.abs(want_xy)) <= 1e-9
    if cfg_name == "tight":
        assert ((wf & abi.FLAG["CURV_ADJUST"]) != 0).sum() > ((g["tr_flags"] & abi.FLAG["CURV_ADJUST"]) != 0).sum()
