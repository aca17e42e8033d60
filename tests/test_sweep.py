"""Candidate sweep (BASELINE config 4, SURVEY §8f-2): 384 candidates per frame through
SpeedController / TrajectoryBuilder, scored on their output points, argmin-selected.

The oracle is "the same loop over the reference's classes": every candidate trajectory is
built by the CPU checker's TrajectoryBuilder (the C restatement, and — CPU test — the
reference's own compiled class), the SpeedController arithmetic and the score are restated
here in numpy from include/pp.h.

Against that loop the GPU sweep runs on both planners under it (warp per frame below 1,536
frames, the pipeline above), on block and warp tails, on rare, resting, cruising and poisoned
frames, on other tracks, configs and car counts, and with held-over cars.  At the benchmark's
size (32,768 frames) the checks need no CPU loop: optional scores, shards, kernel variants,
streams and per-row identities.
"""
import ctypes as C

import numpy as np
import pytest

import checkers

abi = checkers.abi
L, S, T = abi.SWEEP_LANES, abi.SWEEP_SPEEDS, abi.SWEEP_TIMES
M = L * S * T
BAD = abi.SWEEP_BAD
DEFAULT = abi.default_config()
FALLBACK = abi.FLAG["FALLBACK"]
LANES = np.repeat(np.arange(L), S * T).astype(np.int32)   # lane of each candidate index


def candidate_controllers(ego_speed, cfg=DEFAULT):
    """SpeedController(ego_speed) then add_limit_breakpoint(v_i, t_j) (src/main.cpp:493-533)
    for frames of ego speeds `ego_speed` (a scalar or an array) -> (target, time, took), each
    [..., S*T]; `took`: the breakpoint replaced the default controller (ngrade < grade)."""
    e = np.asarray(ego_speed, dtype=np.float64)[..., None]
    v = np.repeat(np.arange(S) * cfg.max_speed / (S - 1), T)
    t = np.tile(0.5 * (np.arange(T) + 1), S)
    target0 = cfg.max_speed
    with np.errstate(invalid="ignore", over="ignore"):
        time0 = np.abs(e - cfg.max_speed) / cfg.relaxed_acc
        grade = (target0 - e) / np.maximum(time0, 0.02)
        ngrade = (v - e) / np.maximum(t, 0.02)
        took = ngrade < grade
    return np.where(took, v, target0), np.where(took, t, time0), took


def score_points(x, y, n, fallback, lane, target_lane, cfg=DEFAULT):
    """include/pp.h: score from the output points alone (same operation order as the kernel)."""
    if fallback or n < 3:
        return abi.SWEEP_BAD
    np.seterr(invalid="ignore")
    vx = (x[1:n] - x[:n - 1]) * 50
    vy = (y[1:n] - y[:n - 1]) * 50
    vsum = np.cumsum(np.sqrt(vx * vx + vy * vy))[-1]   # sequential sum, like the kernel
    ax = (vx[1:] - vx[:-1]) * 50
    ay = (vy[1:] - vy[:-1]) * 50
    amax = np.max(np.sqrt(ax * ax + ay * ay))
    mean = vsum / (n - 1)
    over = amax - cfg.maximum_acc
    over = over if over > 0 else 0.0
    with np.errstate(invalid="ignore"):
        s = abs(float(lane - target_lane)) + (cfg.max_speed - mean) / cfg.max_speed + 0.5 * over
    return s if s < abi.SWEEP_BAD else abi.SWEEP_BAD   # NaN / inf points (e.g. a standstill) are bad


def score_rows(x, y, n, fallback, lane, target_lane, cfg=DEFAULT):
    """score_points over the rows of x, y [m][50] (n, fallback, lane, target_lane: [m]): the
    same operations in the same order, masked by n, so the same bits."""
    m = x.shape[0]
    n = np.broadcast_to(np.asarray(n, dtype=np.int64), (m,))
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        vx = (x[:, 1:] - x[:, :-1]) * 50
        vy = (y[:, 1:] - y[:, :-1]) * 50
        vsum = np.cumsum(np.sqrt(vx * vx + vy * vy), axis=1)   # sequential along each row
        ax = (vx[:, 1:] - vx[:, :-1]) * 50
        ay = (vy[:, 1:] - vy[:, :-1]) * 50
        acc = np.sqrt(ax * ax + ay * ay)
        live = np.arange(acc.shape[1])[None, :] < (n - 2)[:, None]
        amax = np.max(np.where(live, acc, -np.inf), axis=1)
        mean = vsum[np.arange(m), np.clip(n - 2, 0, None)] / (n - 1)
        over = amax - cfg.maximum_acc
        over = np.where(over > 0, over, 0.0)
        s = np.abs((np.asarray(lane) - np.asarray(target_lane)).astype(np.float64)) + \
            (cfg.max_speed - mean) / cfg.max_speed + 0.5 * over
    ok = ~np.asarray(fallback, dtype=bool) & (n >= 3) & (s < BAD)
    return np.where(ok, s, BAD)


def cpu_sweep(chk, frames, plans, cfg=None, rows=None, chunk=64):
    """All candidates of the frames `rows` (default: every frame) through the checker's
    TrajectoryBuilder -> (scores [k][384], (x, y [k][384][50], n_points [k][384]))."""
    rows = np.arange(frames.n) if rows is None else np.asarray(rows)
    k = len(rows)
    scores = np.empty((k, M))
    ox, oy = np.empty((k, M, abi.PATH_LEN)), np.empty((k, M, abi.PATH_LEN))
    on = np.empty((k, M), np.int32)
    for lo in range(0, k, chunk):
        r = rows[lo:lo + chunk]
        c = len(r)
        has_prev = frames.prev_n[r] >= abi.PREV_KEEP
        ex = np.where(has_prev, frames.prev_x[r, -1], frames.ego_x[r])
        ey = np.where(has_prev, frames.prev_y[r, -1], frames.ego_y[r])
        tg, tm, _ = candidate_controllers(plans.ego_speed[r], cfg or DEFAULT)
        rep = lambda a: np.repeat(np.asarray(a), M, axis=0)   # one copy per candidate
        lanes = np.tile(LANES, c)
        x, y, n, fl = chk.trajectory_build(
            rep(frames.prev_n[r]), rep(frames.prev_x[r]), rep(frames.prev_y[r]), rep(ex), rep(ey),
            rep(frames.ego_yaw_deg[r]), lanes, rep(plans.ego_d[r]), rep(plans.ego_vd[r]),
            rep(plans.ego_speed[r]), np.tile(tg, L).ravel(), np.tile(tm, L).ravel(), cfg=cfg)
        scores[lo:lo + c] = score_rows(x, y, n, (fl & FALLBACK) != 0, lanes,
                                       rep(plans.target_lane[r]), cfg or DEFAULT).reshape(c, M)
        ox[lo:lo + c], oy[lo:lo + c] = x.reshape(c, M, -1), y.reshape(c, M, -1)
        on[lo:lo + c] = n.reshape(c, M)
    return scores, (ox, oy, on)


def sweep_paths(want, trajs, plans, frames, cfg=None):
    """What the CPU loop's candidates (every frame) went through: BAD candidates, (frame, lane)s
    whose builder fell back (all 128 BAD), v_0 candidates that stand still (NaN points), rolling
    stops, frames with every candidate BAD."""
    tg, _, _ = candidate_controllers(plans.ego_speed, cfg or DEFAULT)
    bad = want >= BAD
    lane_bad = bad.reshape(len(want), L, S * T).all(axis=2)
    ox, _, on = trajs
    nan_pts = (np.isnan(ox) & (np.arange(abi.PATH_LEN) < on[..., None])).any(axis=2)
    v0 = np.tile(tg, L) == 0
    return dict(frames=len(want), candidates=want.size, bad=int(bad.sum()),
                lanes_bad=int(lane_bad.sum()), v0_standstill=int((nan_pts & v0).sum()),
                rolling_stops=int(rolling_stops(frames, trajs, np.arange(frames.n)).sum()),
                all_bad=int(bad.all(axis=1).sum()))


def test_cpu_sweep_oracle_matches_reference_classes(pp, oracle, ref):
    """The sweep's oracle (C restatement) against the reference's own compiled classes."""
    fb = pp.synth_frames(pp.Map(), 6, 12, seed=404, rare_permille=0)
    plans = oracle.plan(fb, threads=2)
    so, _ = cpu_sweep(oracle, fb, plans)
    sr, _ = cpu_sweep(ref, fb, plans)
    assert np.array_equal(so, sr)
    assert (so < abi.SWEEP_BAD).mean() > 0.9 and np.ptp(so[so < abi.SWEEP_BAD]) > 0.5


def rest_and_cruise_frames(pp, m, n, seed, cfg=DEFAULT):
    """Thirds of n frames, built as in the planner's standstill test (no previous path): at
    rest behind a stopped car 14.7 m ahead, at rest on a free road, and on a free road exactly
    at max_speed."""
    fb = pp.synth_frames(m, n, 12, seed=seed, rare_permille=0)
    a, b = n // 3, 2 * n // 3
    fb.prev_n[:] = 0
    fb.ego_speed_mph[:b] = 0.0
    yaw = np.deg2rad(fb.ego_yaw_deg[:a])
    fb.n_cars[:a] = 1
    fb.car_x[:a, 0] = fb.ego_x[:a] + 14.7 * np.cos(yaw)
    fb.car_y[:a, 0] = fb.ego_y[:a] + 14.7 * np.sin(yaw)
    fb.car_vx[:a, 0] = 0.0
    fb.car_vy[:a, 0] = 0.0
    fb.n_cars[a:] = 0
    mph = cfg.max_speed * 2.237   # a cold start plans with the speed ego_speed_mph / 2.237
    mph = min((np.nextafter(mph, -np.inf), mph, np.nextafter(mph, np.inf)),
              key=lambda v: abs(v / 2.237 - cfg.max_speed))
    assert mph / 2.237 == cfg.max_speed
    fb.ego_speed_mph[b:] = mph
    return fb, (slice(0, a), slice(a, b), slice(b, n))


def poisoned_frames(pp, m, n, seed):
    """NaN / infinite / huge / denormal values in every input field, as in the planner's
    poisoned-fields test -> (frames, mask of frames whose every input is finite)."""
    fb = pp.synth_frames(m, n, 4, seed=seed, rare_permille=0)
    vals = [np.nan, np.inf, -np.inf, 1e200, 1e-310]
    fields = ["car_x", "car_y", "car_vx", "car_vy", "ego_yaw_deg", "ego_speed_mph", "prev_x", "prev_y"]
    for f in range(n):
        a = getattr(fb, fields[(f // 5) % 8])
        if a.ndim == 2:
            a[f, (f // 40) % a.shape[1]] = vals[f % 5]
        else:
            a[f] = vals[f % 5]
    fb.prev_n[::3] = 0
    finite = np.ones(n, bool)
    for k, v in fb.arrays().items():
        if v.dtype == np.float64:
            finite &= np.isfinite(v.reshape(n, -1)).all(axis=1)
    return fb, finite


def test_vectorised_scorer_is_the_scalar_scorer(pp, oracle):
    """score_rows equals score_points bit for bit on planner outputs: rare frames, fallbacks,
    standstills (one NaN point), and every row again with a random n (0, 1, 2 and rows reaching
    into the NaN tail included), under two configs."""
    m = pp.Map()
    fb = pp.synth_frames(m, 300, 12, seed=5, rare_permille=400)
    rest, _ = rest_and_cruise_frames(pp, m, 90, seed=6)
    fb = abi.FrameBatch.concat([fb, rest])
    rng = np.random.default_rng(7)
    hits = dict(nan=0, short=0, fallback=0, standstill=0)
    for cfg in (DEFAULT, checkers.config("tight")):
        plans = oracle.plan(fb, threads=8, cfg=cfg)
        fall = (plans.flags & FALLBACK) != 0
        for n in (plans.n_points, rng.integers(0, abi.PATH_LEN + 1, fb.n)):
            lane = rng.integers(0, L, fb.n)
            got = score_rows(plans.next_x, plans.next_y, n, fall, lane, plans.target_lane, cfg)
            want = np.array([score_points(plans.next_x[f], plans.next_y[f], int(n[f]), bool(fall[f]),
                                          int(lane[f]), int(plans.target_lane[f]), cfg)
                             for f in range(fb.n)])
            assert np.array_equal(got.view(np.int64), want.view(np.int64))
            hits["nan"] += int(np.isnan(plans.next_x[np.arange(fb.n), np.maximum(n - 1, 0)]).sum())
            hits["short"] += int((n < 3).sum())
            hits["fallback"] += int(fall.sum())
        hits["standstill"] += int(((plans.n_points == 1) & np.isnan(plans.next_x[:, 0])).sum())
    assert min(hits.values()) > 0, hits


# ---- the GPU sweep against the CPU loop -------------------------------------------------------

@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def gmap(pp, torch_cuda):
    return pp.Map()


def run_sweep(pp, torch, m, fb, cfg=None, want_scores=True):
    """pp_sweep_batch -> (dict of numpy arrays, launches it made)."""
    df = pp.DeviceFrames(fb)
    before = pp.launch_count()
    out = pp.sweep_batch(m, df, cfg=cfg, want_scores=want_scores)
    torch.cuda.synchronize()
    launches = pp.launch_count() - before
    return {k: v.cpu().numpy() for k, v in out.items() if v is not None}, launches


def rolling_stops(frames, trajs, rows):
    """[k][384]: candidates whose CPU trajectory slows to a standstill after moving (a step of
    zero or NaN length right after a moving one, among the newly emitted points).  At that
    point the reference's chord division is 0 * 0 / |chord| with a chord of rounding size
    (~1e-19 m): the last bit of the spline value or of the running position, both well inside
    the 1e-9 trajectory bar, decides between a finite point (the car stays put) and the 0/0 NaN
    that makes the candidate BAD.  A standstill from rest (a 0/0 at the first point) is not
    one of these."""
    ox, oy, on = trajs
    with np.errstate(invalid="ignore"):
        d = np.hypot(np.diff(ox, axis=2), np.diff(oy, axis=2))        # d[i]: point i -> i + 1
    i = np.arange(abi.PATH_LEN - 1)
    kept = np.where(frames.prev_n[rows] >= abi.PREV_KEEP, abi.PREV_KEEP, 0)[:, None, None]
    live = i < on[..., None] - 1
    moving = live & (d > 0)
    stop = live & ~(d > 0) & (i >= kept)
    return (stop[..., 1:] & moving[..., :-1]).any(axis=2)


def check_sweep_against_cpu_loop(pp, oracle, fb=None, cfg=None, m=None, want_scores=True,
                                 rows=None, full=None, diverse=False):
    """pp_sweep_batch on `fb` (default: 96 synthetic frames, 12 cars, seed 77, 120 permille rare)
    over the device map `m` (default: the highway; `oracle` must hold the same track) with `cfg`
    (None: the defaults) against cpu_sweep with the same config, on the frames `rows` (default:
    all).  The full bars hold on the rows where `full` (default: all) is set; on the others the
    BAD pattern, the winner and its point count still equal the CPU's.  Rolling stops (see
    rolling_stops) may come out BAD on one side only, in at most 2 % of them (plus 2).
    Returns (CPU scores, CPU trajectories, CPU plans, GPU outputs, launches)."""
    import torch
    m = m if m is not None else pp.Map()
    if fb is None:
        fb = pp.synth_frames(m, 96, 12, seed=77, rare_permille=120)
    n = fb.n
    rows = np.arange(n) if rows is None else np.asarray(rows)
    full = np.ones(len(rows), bool) if full is None else np.asarray(full)[rows]
    plans = oracle.plan(fb, threads=8, cfg=cfg)
    want, trajs = cpu_sweep(oracle, fb, plans, cfg, rows=rows)
    out, launches = run_sweep(pp, torch, m, fb, cfg, want_scores)
    best, best_score = out["best"][rows], out["best_score"][rows]
    k = np.arange(len(rows))
    bad_w = want >= BAD
    stops = rolling_stops(fb, trajs, rows)
    if want_scores:
        got = out["scores"][rows]
        flip = bad_w != (got >= BAD)
        assert not (flip & ~stops).any(), np.argwhere(flip & ~stops)[:5].tolist()
        assert flip.sum() <= 0.02 * stops.sum() + 2, (int(flip.sum()), int(stops.sum()))
        ok = ~bad_w & ~flip & full[:, None]
        if ok.any():  # trajectories agree to ~1e-13 m; A_k = d2P * 2500
            assert np.max(np.abs(got[ok] - want[ok])) <= 1e-6
        assert np.array_equal(best, np.argmin(got, axis=1))            # lowest score, lowest index on ties
        assert np.array_equal(best_score.view(np.int64), got[k, best].view(np.int64))
    else:
        flip = stops   # which of them flipped is not known without the scores
        sure = ~flip.any(axis=1)
        assert np.array_equal((best_score >= BAD)[sure], bad_w.all(axis=1)[sure])
        live = (best_score < BAD) & ~flip[k, best] & full
        assert np.max(np.abs(best_score[live] - want[k, best][live]), initial=0) <= 1e-6
    opt = np.where(flip, BAD, want)   # the oracle's scores where both sides agree on BAD
    mine = ~flip[k, best] & full
    assert (want[k, best][mine] <= opt.min(axis=1)[mine] + 1e-6).all()  # ... and it is the oracle's optimum
    if full.sum() >= 20:
        assert (best == np.argmin(opt, axis=1))[full].mean() > 0.95
    assert np.array_equal(best[~full], np.argmin(opt, axis=1)[~full])
    # the returned trajectory is the winning candidate's
    nx, ny, npts = out["next_x"][rows], out["next_y"][rows], out["n_points"][rows]
    ox, oy, on = trajs
    for i in range(len(rows)):
        assert np.isnan(nx[i, npts[i]:]).all() and np.isnan(ny[i, npts[i]:]).all()
        if best_score[i] >= BAD:
            assert npts[i] == 0
            continue
        c = best[i]
        if flip[i, c]:
            continue
        assert npts[i] == on[i, c]
        if full[i]:
            assert np.allclose(nx[i, :npts[i]], ox[i, c, :npts[i]], rtol=1e-9, atol=1e-6)
            assert np.allclose(ny[i, :npts[i]], oy[i, c, :npts[i]], rtol=1e-9, atol=1e-6)
    if diverse:  # the sweep really differentiates: several lanes and speeds win somewhere
        assert len(np.unique(best // (S * T))) >= 2 and len(np.unique(best)) > 5
    return want, trajs, plans, out, launches


@pytest.mark.gpu
def test_sweep_matches_cpu_loop(pp, torch_cuda, oracle):
    check_sweep_against_cpu_loop(pp, oracle, diverse=True)


@pytest.mark.gpu
def test_sweep_follows_the_config(pp, torch_cuda, oracle):
    """Candidates and scores follow the config: speeds up to max_speed, time from relaxed_acc,
    the acceleration penalty above maximum_acc, and the planning step's ego state (the tight
    config moves every tunable)."""
    want, _, plans, _, _ = check_sweep_against_cpu_loop(pp, oracle, cfg=checkers.config("tight"),
                                                        diverse=True)
    fb = pp.synth_frames(pp.Map(), 96, 12, seed=77, rare_permille=120)
    base, _ = cpu_sweep(oracle, fb, oracle.plan(fb, threads=8))
    ok = (want < abi.SWEEP_BAD) & (base < abi.SWEEP_BAD)
    assert (want[ok] != base[ok]).mean() > 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 5, 7, 97])
def test_sweep_block_and_warp_tails(pp, torch_cuda, gmap, oracle, n):
    """Batches that end inside a select block (4 frames per block) and a warp: every frame,
    the last one included, is scored, selected and emitted."""
    fb = pp.synth_frames(gmap, n, 12, seed=77, rare_permille=120)
    check_sweep_against_cpu_loop(pp, oracle, fb, m=gmap)


@pytest.mark.gpu
@pytest.mark.parametrize("n,want_scores", [(1535, True), (1537, True), (4100, False)])
def test_sweep_on_both_planners(pp, torch_cuda, gmap, oracle, n, want_scores):
    """Around the planner's switch at 1,536 frames: the warp-per-frame kernel below, the
    pipeline above (the benchmark's planner, with the sweep's mix of NULL and set plan outputs),
    compared on a strided sample of ~200 frames and the last frame; 4,100 frames take the
    benchmark's output path, without scores."""
    fb = pp.synth_frames(gmap, n, 12, seed=1000 + n, rare_permille=120)
    rows = np.unique(np.r_[np.arange(0, n, n // 200), n - 1])
    *_, launches = check_sweep_against_cpu_loop(pp, oracle, fb, m=gmap, rows=rows,
                                                want_scores=want_scores, diverse=True)
    if n < 1536:
        assert launches == 1 + 3   # plan_warp, then setup / emit / select
    else:
        assert launches > 1 + 3    # the pipeline: three launches per chunk


@pytest.mark.gpu
def test_sweep_on_rare_frames(pp, torch_cuda, gmap, oracle):
    """rare_permille = 1000: every frame is one of pp_synth.cu's rare kinds (standstill, crawl,
    cold start, ego lost, on a waypoint, hard brake, follow, collision, off-road, ...)."""
    fb = pp.synth_frames(gmap, 300, 12, seed=78, rare_permille=1000)
    assert set(np.unique(fb.prev_n)) >= {0, 3, 9}           # cold starts of every length
    still = (fb.prev_n >= abi.PREV_KEEP) & (fb.prev_x == fb.prev_x[:, :1]).all(axis=1)
    assert still.sum() >= 10                                 # standstills: one repeated point
    want, trajs, plans, _, _ = check_sweep_against_cpu_loop(pp, oracle, fb, m=gmap)
    paths = sweep_paths(want, trajs, plans, fb)
    assert paths["v0_standstill"] > 0 and paths["lanes_bad"] > 0 and paths["all_bad"] > 0, paths
    assert ((plans.flags & abi.FLAG["EGO_MATCH_FAIL"]) != 0).sum() > 0


@pytest.mark.gpu
def test_sweep_at_rest_and_cruise(pp, torch_cuda, gmap, oracle):
    """At rest (behind a stopped car, or on a free road) a v_0 candidate has a zero arc step
    and a 0/0 chord, the planner's single NaN point: the emission kernel's lean loop hands it
    to the complete one (bail 5), which must come out BAD, while every other candidate stays
    finite.  Cruising exactly at max_speed gives the default controller time0 = 0 (a ramp that
    is over before it starts), which must stay finite."""
    fb, (stopped, free, cruise) = rest_and_cruise_frames(pp, gmap, 300, seed=79)
    want, trajs, plans, out, _ = check_sweep_against_cpu_loop(pp, oracle, fb, m=gmap)
    tg, tm, took = candidate_controllers(plans.ego_speed, DEFAULT)
    v0 = np.tile(tg == 0, L)   # [n][384]: the candidate's target speed is 0
    built = np.repeat(want.reshape(fb.n, L, S * T).min(axis=2) < BAD, S * T, axis=1)  # lane not fallen back
    for part in (stopped, free):
        assert (plans.ego_speed[part] == 0).all()
        assert v0[part].sum(axis=1).min() == L * T   # every v_0 candidate targets 0
        assert (want[part][v0[part] & built[part]] >= BAD).all()
        assert (want[part][~v0[part] & built[part]] < BAD).all()
        assert built[part].mean() > 0.9
    assert (plans.ego_speed[cruise] == DEFAULT.max_speed).all()
    assert (tm[cruise][~took[cruise]] == 0).all() and (~took[cruise]).sum() > 0   # time0 = 0
    assert (want[cruise][np.tile(~took[cruise], L) & built[cruise]] < BAD).all()
    assert (out["best_score"] < BAD).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n_wp", [("circle", 40), ("ellipse", 400), ("circle", 7)])
def test_sweep_on_other_maps(pp, torch_cuda, kind, n_wp):
    """The tracks of the planner's test_other_maps: k_sweep_setup builds its own map view
    (pad_lo = min(n_wp, PPD_PAD)), so a short loop, a long one and a 7-point loop."""
    th = np.linspace(0.0, 2 * np.pi, n_wp, endpoint=False)
    if kind == "circle":
        r = 40.0 * n_wp / (2 * np.pi)
        wx, wy = 1000 + r * np.cos(-th), 2000 + r * np.sin(-th)
    else:
        wx, wy = 3000 + 2400 * np.cos(-th), 1000 + 1100 * np.sin(-th)
    chk = checkers.Checker("oracle")
    chk.map_from_points(wx, wy)
    m = pp.Map(points=(wx, wy))
    assert np.array_equal(m.table(), chk.map_table())
    fb = pp.synth_frames(m, 200, 12, seed=n_wp, rare_permille=100)
    check_sweep_against_cpu_loop(pp, chk, fb, m=m)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name", ["loose", "max25", "edges"])
def test_sweep_under_other_configs(pp, torch_cuda, gmap, oracle, cfg_name):
    cfg = checkers.config(cfg_name)
    fb = pp.synth_frames(gmap, 200, 12, seed=80, rare_permille=120)
    want, _, plans, out, _ = check_sweep_against_cpu_loop(pp, oracle, fb, cfg=cfg, m=gmap)
    if cfg_name == "loose":   # candidates reach 40 m/s, and some win
        tg, _, _ = candidate_controllers(plans.ego_speed, cfg)
        won = np.tile(tg, L)[np.arange(fb.n), out["best"]]
        assert (won[out["best_score"] < BAD] > 30).any()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["0 cars", "1 car", "64 cars", "ragged", "held over"])
def test_sweep_car_counts(pp, torch_cuda, gmap, oracle, case):
    """The cars enter the sweep through the planner's target lane, which enters every score:
    no car, one, 64, ragged n_cars, and cars held over from an earlier message (planned on the
    CPU with the same frozen arrays)."""
    cars = {"0 cars": 0, "1 car": 1, "64 cars": 64}.get(case, 12)
    rng = np.random.default_rng(cars)
    fb = pp.synth_frames(gmap, 200, cars, seed=81 + cars, rare_permille=100, max_cars=max(cars, 1))
    if case in ("ragged", "held over"):
        fb.n_cars[::3] = rng.integers(0, cars + 1, len(fb.n_cars[::3]))
    if case == "held over":
        fb, pick = checkers.hold_over(fb, oracle.plan(fb, threads=8), rng)
        assert pick.sum() > 100
    _, _, plans, _, _ = check_sweep_against_cpu_loop(pp, oracle, fb, m=gmap)
    if cars:
        assert (plans.target_lane != plans.ego_lane).any()


@pytest.mark.gpu
def test_sweep_on_poisoned_fields(pp, torch_cuda, gmap, oracle):
    """NaN / infinite / huge / denormal inputs: the sweep returns; BAD pattern, winner and point
    count equal the CPU's everywhere, the full bars hold where every input is finite."""
    fb, finite = poisoned_frames(pp, gmap, 400, seed=92)
    assert 0.2 < finite.mean() < 0.6
    check_sweep_against_cpu_loop(pp, oracle, fb, m=gmap, full=finite)


# ---- the benchmark's size: GPU against itself -------------------------------------------------

BENCH_N, BENCH_SEED = 32768, 0x5EED   # bench.py --workload sweep: 32,768 frames, 12 cars


@pytest.fixture(scope="module")
def bench_case(pp, torch_cuda, gmap):
    """The benchmark's frames and their sweep with scores."""
    fb = pp.synth_frames(gmap, BENCH_N, 12, seed=BENCH_SEED)
    out, launches = run_sweep(pp, torch_cuda, gmap, fb)
    assert launches > 1 + 3
    return fb, out


def assert_same(a, b, keys=None):
    for k in keys or a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
        if a[k].dtype == np.float64:   # bit for bit, NaN payloads aside
            x, y = a[k].view(np.int64), b[k].view(np.int64)
            assert np.array_equal(x[~np.isnan(a[k])], y[~np.isnan(b[k])]), k


@pytest.mark.gpu
def test_bench_size_without_scores(pp, torch_cuda, gmap, bench_case):
    """want_scores=False (the benchmark's call) returns the same winner, bit for bit."""
    fb, full = bench_case
    lean, _ = run_sweep(pp, torch_cuda, gmap, fb, want_scores=False)
    assert "scores" not in lean
    assert_same(lean, full, ("best", "best_score", "next_x", "next_y", "n_points"))


@pytest.mark.gpu
def test_bench_size_shards(pp, torch_cuda, gmap, bench_case):
    """The whole batch (pipeline planner) equals sweeps over chunks of 1,000 frames (warp
    planner), concatenated, scores included."""
    fb, full = bench_case
    parts = [run_sweep(pp, torch_cuda, gmap, fb.slice(lo, min(lo + 1000, fb.n)))[0]
             for lo in range(0, fb.n, 1000)]
    assert_same({k: np.concatenate([p[k] for p in parts]) for k in full}, full)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2, 3, 4])
def test_bench_size_kernel_variants(pp, torch_cuda, gmap, bench_case, variant):
    """Every planner variant under the sweep gives the same bits."""
    fb, full = bench_case
    pp.set_kernel_variant(variant)
    try:
        got, _ = run_sweep(pp, torch_cuda, gmap, fb)
    finally:
        pp.set_kernel_variant(0)
    assert_same(got, full)


@pytest.mark.gpu
def test_bench_size_row_identities(pp, torch_cuda, gmap, bench_case):
    """Per row: best_score = min(scores) at its lowest index; no points exactly when the winner
    is BAD; NaN beyond n_points; the kept previous points lead the path; and within a
    (frame, lane) the candidates left with the default controller score the same bits."""
    fb, out = bench_case
    n = fb.n
    s, best, bs, npts = out["scores"], out["best"], out["best_score"], out["n_points"]
    assert np.array_equal(bs, s.min(axis=1)) and np.array_equal(best, np.argmin(s, axis=1))
    assert np.array_equal(npts == 0, bs >= BAD)
    assert (bs < BAD).mean() > 0.95
    tail = np.arange(abi.PATH_LEN)[None, :] >= npts[:, None]
    assert np.isnan(out["next_x"][tail]).all() and np.isnan(out["next_y"][tail]).all()
    assert not np.isnan(out["next_x"][~tail]).any()
    kept = (fb.prev_n >= abi.PREV_KEEP) & (npts > 0)
    assert kept.mean() > 0.9
    assert np.array_equal(out["next_x"][kept, :abi.PREV_KEEP], fb.prev_x[kept])
    assert np.array_equal(out["next_y"][kept, :abi.PREV_KEEP], fb.prev_y[kept])
    dp = pp.DevicePlans(n, fb.max_cars, diag=True, cars=False)
    pp.plan_batch(gmap, pp.DeviceFrames(fb), dp)
    torch_cuda.cuda.synchronize()
    _, _, took = candidate_controllers(dp.to_host().ego_speed)
    dflt = np.repeat(~took[:, None, :], L, axis=1)            # [n][lane][128]
    s3 = s.reshape(n, L, S * T)
    hi = np.where(dflt, s3, -np.inf).max(axis=2)
    lo = np.where(dflt, s3, np.inf).min(axis=2)
    some = dflt.any(axis=2)
    assert some.mean() > 0.5
    assert np.array_equal(hi[some], lo[some])


@pytest.mark.gpu
def test_sweep_on_a_side_stream(pp, torch_cuda, gmap, bench_case):
    """Issued on a non-default stream, the sweep gives the default stream's result."""
    fb, full = bench_case
    torch = torch_cuda
    df = pp.DeviceFrames(fb)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        out = pp.sweep_batch(gmap, df)
    side.synchronize()
    assert_same({k: v.cpu().numpy() for k, v in out.items()}, full)


# ---- argument handling -----------------------------------------------------------------------

@pytest.mark.gpu
def test_sweep_rejects_bad_arguments(pp, torch_cuda, gmap):
    """PP_E_ARG (-1) for each NULL required output and for n < 0; n = 0 returns 0 and writes
    nothing."""
    torch = torch_cuda
    n = 8
    fb = pp.synth_frames(gmap, n, 12, seed=3)
    df = pp.DeviceFrames(fb)
    bufs = {"best": torch.full((n,), -7, dtype=torch.int32, device="cuda"),
            "best_score": torch.full((n,), -7.0, dtype=torch.float64, device="cuda"),
            "next_x": torch.full((n, abi.PATH_LEN), -7.0, dtype=torch.float64, device="cuda"),
            "next_y": torch.full((n, abi.PATH_LEN), -7.0, dtype=torch.float64, device="cuda"),
            "n_points": torch.full((n,), -7, dtype=torch.int32, device="cuda"),
            "scores": torch.full((n, M), -7.0, dtype=torch.float64, device="cuda")}
    cfg, fs = abi.default_config(), df.struct()

    def call(count, drop=None):
        so = abi.SweepOut()
        for k, v in bufs.items():
            setattr(so, k, None if k == drop else v.data_ptr())
        rc = pp.lib.pp_sweep_batch(gmap.handle, C.byref(cfg), C.byref(fs), C.byref(so),
                                   C.c_int64(count), None)
        torch.cuda.synchronize()
        return rc

    for k in ("best", "best_score", "next_x", "next_y", "n_points"):
        assert call(n, drop=k) == -1, k
    assert call(-1) == -1
    assert call(0) == 0
    for k, v in bufs.items():
        assert (v == -7).all(), k
    assert call(n, drop="scores") == 0   # scores are optional
    assert (bufs["scores"] == -7).all() and (bufs["n_points"] >= 0).all()
