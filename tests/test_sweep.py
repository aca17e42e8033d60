"""Candidate sweep (BASELINE config 4, SURVEY §8f-2): 384 candidates per frame through
SpeedController / TrajectoryBuilder, scored on their output points, argmin-selected.

The oracle is "the same loop over the reference's classes": every candidate trajectory is
built by the CPU checker's TrajectoryBuilder (the C restatement, and — CPU test — the
reference's own compiled class), the SpeedController arithmetic and the score are restated
here in numpy from include/pp.h.
"""
import numpy as np
import pytest

import checkers

abi = checkers.abi
L, S, T = abi.SWEEP_LANES, abi.SWEEP_SPEEDS, abi.SWEEP_TIMES
DEFAULT = abi.default_config()


def candidate_controllers(ego_speed, cfg=DEFAULT):
    """SpeedController(ego_speed) then add_limit_breakpoint(v_i, t_j) (src/main.cpp:493-533)
    for one frame -> (target[S*T], time[S*T])."""
    target0 = cfg.max_speed
    time0 = abs(ego_speed - cfg.max_speed) / cfg.relaxed_acc
    tg, tm = np.empty(S * T), np.empty(S * T)
    for iv in range(S):
        for it in range(T):
            v, t = iv * cfg.max_speed / (S - 1), 0.5 * (it + 1)
            grade = (target0 - ego_speed) / max(time0, 0.02)
            ngrade = (v - ego_speed) / max(t, 0.02)
            take = ngrade < grade
            tg[iv * T + it] = v if take else target0
            tm[iv * T + it] = t if take else time0
    return tg, tm


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


def cpu_sweep(chk, frames, plans, cfg=None):
    """All candidates of every frame through the checker's TrajectoryBuilder."""
    n = frames.n
    scores = np.empty((n, abi.SWEEP_CANDS))
    trajs = {}
    for f in range(n):
        has_prev = frames.prev_n[f] >= abi.PREV_KEEP
        ex = frames.prev_x[f, -1] if has_prev else frames.ego_x[f]
        ey = frames.prev_y[f, -1] if has_prev else frames.ego_y[f]
        tg, tm = candidate_controllers(plans.ego_speed[f], cfg or DEFAULT)
        m = L * S * T
        rep = lambda a: np.repeat(np.asarray(a)[None], m, axis=0)
        lanes = np.repeat(np.arange(L), S * T).astype(np.int32)
        ox, oy, on, fl = chk.trajectory_build(
            rep(frames.prev_n[f]).astype(np.int32), rep(frames.prev_x[f]), rep(frames.prev_y[f]),
            rep(ex), rep(ey), rep(frames.ego_yaw_deg[f]), lanes, rep(plans.ego_d[f]),
            rep(plans.ego_vd[f]), rep(plans.ego_speed[f]), np.tile(tg, L), np.tile(tm, L), cfg=cfg)
        for c in range(m):
            fb = bool(fl[c] & abi.FLAG["FALLBACK"])
            scores[f, c] = score_points(ox[c], oy[c], int(on[c]), fb, int(lanes[c]),
                                        int(plans.target_lane[f]), cfg or DEFAULT)
        trajs[f] = (ox, oy, on)
    return scores, trajs


def test_cpu_sweep_oracle_matches_reference_classes(pp, oracle, ref):
    """The sweep's oracle (C restatement) against the reference's own compiled classes."""
    fb = pp.synth_frames(pp.Map(), 6, 12, seed=404, rare_permille=0)
    plans = oracle.plan(fb, threads=2)
    so, _ = cpu_sweep(oracle, fb, plans)
    sr, _ = cpu_sweep(ref, fb, plans)
    assert np.array_equal(so, sr)
    assert (so < abi.SWEEP_BAD).mean() > 0.9 and np.ptp(so[so < abi.SWEEP_BAD]) > 0.5


def check_sweep_against_cpu_loop(pp, oracle, cfg=None):
    """pp_sweep_batch with `cfg` (None: the defaults) against cpu_sweep with the same config;
    returns (frames, CPU scores)."""
    n = 96
    m = pp.Map()
    fb = pp.synth_frames(m, n, 12, seed=77, rare_permille=120)
    plans = oracle.plan(fb, threads=8, cfg=cfg)
    want, trajs = cpu_sweep(oracle, fb, plans, cfg)
    out = pp.sweep_batch(m, pp.DeviceFrames(fb), cfg=cfg)
    got = out["scores"].cpu().numpy()
    bad_w, bad_g = want >= abi.SWEEP_BAD, got >= abi.SWEEP_BAD
    assert np.array_equal(bad_w, bad_g)
    ok = ~bad_w
    assert np.max(np.abs(got[ok] - want[ok])) <= 1e-6  # trajectories agree to ~1e-13 m; A_k = d2P * 2500
    best = out["best"].cpu().numpy()
    best_score = out["best_score"].cpu().numpy()
    assert np.array_equal(best, np.argmin(got, axis=1))            # lowest score, lowest index on ties
    assert np.array_equal(best_score, got[np.arange(n), best])
    assert (want[np.arange(n), best] <= want.min(axis=1) + 1e-6).all()  # ... and it is the oracle's optimum
    assert (best == np.argmin(want, axis=1)).mean() > 0.95
    # the returned trajectory is the winning candidate's
    nx, ny, npts = out["next_x"].cpu().numpy(), out["next_y"].cpu().numpy(), out["n_points"].cpu().numpy()
    for f in range(n):
        if best_score[f] >= abi.SWEEP_BAD:
            assert npts[f] == 0
            continue
        ox, oy, on = trajs[f]
        c = best[f]
        assert npts[f] == on[c]
        assert np.allclose(nx[f, :npts[f]], ox[c, :npts[f]], rtol=1e-9, atol=1e-6)
        assert np.allclose(ny[f, :npts[f]], oy[c, :npts[f]], rtol=1e-9, atol=1e-6)
        assert np.isnan(nx[f, npts[f]:]).all()
    # the sweep really differentiates: several lanes and speeds win somewhere
    assert len(np.unique(best // (S * T))) >= 2 and len(np.unique(best)) > 5
    return fb, want


@pytest.mark.gpu
def test_sweep_matches_cpu_loop(pp, oracle):
    check_sweep_against_cpu_loop(pp, oracle)


@pytest.mark.gpu
def test_sweep_follows_the_config(pp, oracle):
    """Candidates and scores follow the config: speeds up to max_speed, time from relaxed_acc,
    the acceleration penalty above maximum_acc, and the planning step's ego state (the tight
    config moves every tunable)."""
    fb, want = check_sweep_against_cpu_loop(pp, oracle, checkers.config("tight"))
    base, _ = cpu_sweep(oracle, fb, oracle.plan(fb, threads=8))
    ok = (want < abi.SWEEP_BAD) & (base < abi.SWEEP_BAD)
    assert (want[ok] != base[ok]).mean() > 0.9
