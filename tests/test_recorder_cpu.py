"""The flight recorder of the rollouts (include/pp.h, pp_rollouts_set_recorder) without a GPU: the
constants and the struct of abi.py against pp.h, the argument checks that need no device, the
trigger-name helper, and a recorded window replanned by the CPU oracle (tests/golden/)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import checkers
import recorder_replay

abi = checkers.abi
HERE = os.path.dirname(os.path.abspath(__file__))
PP_H = open(os.path.join(os.path.dirname(HERE), "include", "pp.h")).read()
FIXTURE = os.path.join(HERE, "golden", "recorder_window_c64.npz")


def test_constants_and_struct_match_pp_h():
    assert re.search(r"#define PP_REC_NONFINITE PP_INC_KINDS\b", PP_H)
    assert abi.REC_NONFINITE == abi.INC_KINDS == len(abi.REC_NAMES) - 1
    assert int(re.search(r"#define PP_REC_MAX_WINDOW (\d+)", PP_H).group(1)) == abi.REC_MAX_WINDOW
    body = re.search(r"typedef struct pp_rollout_recording \{(.*?)\} pp_rollout_recording;", PP_H,
                     re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    ctype = {"int64_t": np.int64, "uint32_t": np.uint32, "int32_t": np.int32, "double": np.float64}
    declared = [(n, ctype[t]) for t, group in re.findall(r"(\w+)\s+([^;]+);", body)
                for n in re.findall(r"\*\s*(\w+)", group)]
    assert declared == [(n, dt) for n, dt, _ in abi.REC_FIELDS]
    assert [f for f, _ in abi.RolloutRecording._fields_] == [n for n, _ in declared]
    assert C.sizeof(abi.RolloutRecording) == 8 * len(declared)


def test_trigger_names_to_mask():
    assert abi.rec_mask(0) == 0 and abi.rec_mask(0x55) == 0x55
    assert abi.rec_mask(["collision_front"]) == 1
    assert abi.rec_mask(["nonfinite"]) == 1 << abi.REC_NONFINITE == 1 << 7
    but_rear = [k for k in abi.INC_NAMES if k != "collision_rear"]
    assert abi.rec_mask(but_rear) == 0b1111101
    assert abi.rec_mask(abi.REC_NAMES) == (1 << (abi.REC_NONFINITE + 1)) - 1
    assert abi.rec_mask(("off_road", "off_road")) == 1 << abi.INC["off_road"]
    with pytest.raises(ValueError):
        abi.rec_mask(["collision"])


def test_argument_checks_without_a_device(pp):
    arg = -1  # PP_E_ARG
    lib = pp.lib
    assert lib.pp_rollouts_set_recorder(None, C.c_int32(4), C.c_uint32(0)) == arg
    rec = abi.RolloutRecording()
    assert lib.pp_rollouts_get_recording(None, None, C.c_int64(0), C.byref(rec)) == arg
    assert "pp_rollouts_set_recorder" in pp.EXPORTS and "pp_rollouts_get_recording" in pp.EXPORTS



def _fixture():
    z = np.load(FIXTURE)
    tick = z["tick"][None, :]
    w = tick.shape[1]
    fb = abi.FrameBatch(w, z["in_car_x"].shape[1])
    for k in fb.arrays():
        setattr(fb, k, np.ascontiguousarray(z["in_" + k]))
    dev = abi.PlanBatch(w, fb.max_cars, diag=False, cars=False)
    for k in ("next_x", "next_y", "n_points", "target_lane", "flags"):
        setattr(dev, k, np.ascontiguousarray(z["dev_" + k]))
    return z, fb, dev, tick, z["consume_k"][None, :]


def test_recorded_window_replays_on_the_oracle(oracle):
    """A 64-car IDM window that ends in a non-finite distance (profiles/rollout_recorder.py
    --cars 64 --traffic idm --fixture-out): the device's plans of it close the loop bit for bit,
    and the oracle, replanning its finite frames, reproduces the recorded next frames."""
    z, fb, dev, tick, ck = _fixture()
    filled = tick[0] >= 0
    ok, applies = recorder_replay.closure(fb, dev, tick, ck)
    assert applies.sum() == filled.sum() - 1 and ok[applies].all()
    rows = np.flatnonzero(filled & recorder_replay.frame_finite(fb))
    sub = abi.FrameBatch(len(rows), fb.max_cars)
    for k in fb.arrays():
        setattr(sub, k, np.ascontiguousarray(getattr(fb, k)[rows]))
    cpu = oracle.plan(sub, threads=4, diag=False, cars=False)
    full = abi.PlanBatch(fb.n, fb.max_cars, diag=False, cars=False)
    for k in full.fields:
        getattr(full, k)[...] = getattr(dev, k)
        getattr(full, k)[rows] = getattr(cpu, k)
    ok_cpu, _ = recorder_replay.closure(fb, full, tick, ck, 1e-9, 1e-6)
    assert ok_cpu[applies].all(), np.flatnonzero(~ok_cpu[0] & applies[0])[:5]
    mask = np.zeros((1, fb.n), bool)
    mask[0, rows] = True
    # the fixture keeps the plans' n_points, target_lane and flags, not ego_lane / ref_wp
    assert recorder_replay.oracle_agrees(dev, full, 1, fb.n, mask,
                                         ("n_points", "target_lane", "flags")).all()
    # the planner makes the first non-finite point from a finite frame, and so does the oracle
    first_bad = next(i for i in range(fb.n) if np.isnan(dev.next_x[i, :dev.n_points[i]]).any())
    assert first_bad in rows and np.isnan(full.next_x[first_bad, :full.n_points[first_bad]]).any()
    assert int(z["trigger_tick"]) == tick[0, first_bad] + 10
