import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)

GOLDEN = os.path.join(HERE, "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _ensure_built():
    """Build the product library and the CPU checkers if they are stale/missing
    (the driver normally runs __graft_entry__.build() first; this keeps a bare
    `pytest` working too)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "pp_build", os.path.join(ROOT, "carnd-path-planning-project_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True,
                   capture_output=True)


_ensure_built()

import checkers  # noqa: E402


@pytest.fixture(scope="session")
def pp():
    return checkers.load_pkg()


@pytest.fixture(scope="session")
def abi():
    return checkers.abi


@pytest.fixture(scope="session")
def oracle():
    return checkers.Checker("oracle")


@pytest.fixture(scope="session")
def ref():
    if not checkers.available("ref"):
        pytest.skip("oracle/_ref/libppref.so not present (reference sources unavailable)")
    return checkers.Checker("ref")


@pytest.fixture(scope="session")
def pmap(pp):
    return pp.Map()


@pytest.fixture(scope="session")
def golden_units():
    return np.load(os.path.join(GOLDEN, "units.npz"))


def load_golden_frames(abi, tag):
    z = np.load(os.path.join(GOLDEN, f"frames_{tag}.npz"))
    n, mc = z["in_car_x"].shape
    fb = abi.FrameBatch(n, mc)
    for k in fb.arrays():
        setattr(fb, k, np.ascontiguousarray(z["in_" + k]))
    zo = np.load(os.path.join(GOLDEN, f"frames_{tag}_out.npz"))
    outs = {k[4:]: zo[k] for k in zo.files}
    return fb, outs, int(z["observable_flags"])


@pytest.fixture(scope="session", params=["c12", "c64"])
def golden_frames(request, abi):
    return load_golden_frames(abi, request.param)


# ---- comparison helpers shared by the CPU and GPU parity tests ------------

# Fields built only from + - * / sqrt and comparisons: must be bit-identical.
EXACT_F64 = ["ego_s", "ego_d", "ego_vs", "ego_vd", "ego_speed", "ego_acc", "target_speed",
             "target_time", "car_s", "car_d", "car_vs", "car_vd"]
EXACT_INT = ["n_points", "ego_lane", "ref_wp", "target_lane", "next_car_id",
             "next_car_in_target_lane", "car_lane", "car_next_wp"]
# Trajectory points pass through atan2/sin/cos (libm vs CUDA differ by ulps):
# north_star tolerance 1e-9 relative / 1e-6 m absolute.
TRAJ_RTOL = 1e-9
TRAJ_ATOL = 1e-6


def assert_plans_equal(got, want, flag_mask, bitwise_traj, what=""):
    """got / want: dict name -> ndarray.  Integer and exact-f64 fields must be
    identical; next_x/next_y identical (bitwise_traj) or within tolerance."""
    for k in EXACT_INT:
        if k in got and k in want and got[k] is not None and want[k] is not None:
            bad = np.argwhere(got[k] != want[k])
            assert len(bad) == 0, f"{what}{k}: {len(bad)} mismatches, first {bad[:5].tolist()}"
    for k in EXACT_F64:
        if k in got and k in want and got[k] is not None and want[k] is not None:
            a, b = got[k], want[k]
            bad = np.argwhere(~((a == b) | ((a != a) & (b != b))))
            assert len(bad) == 0, (f"{what}{k}: {len(bad)} mismatches, first {bad[:5].tolist()} "
                                   f"{a[tuple(bad[0])]!r} vs {b[tuple(bad[0])]!r}")
    gf, wf = got["flags"] & flag_mask, want["flags"] & flag_mask
    bad = np.argwhere(gf != wf)
    assert len(bad) == 0, (f"{what}flags: {len(bad)} mismatches, first {bad[:5].tolist()} "
                           f"{gf[bad[0][0]]:#x} vs {wf[bad[0][0]]:#x}")
    for k in ("next_x", "next_y"):
        a, b = got[k], want[k]
        nan_a, nan_b = a != a, b != b
        assert np.array_equal(nan_a, nan_b), f"{what}{k}: NaN pattern differs"
        if bitwise_traj:
            bad = np.argwhere(~((a == b) | (nan_a & nan_b)))
            assert len(bad) == 0, f"{what}{k}: {len(bad)} mismatches, first {bad[:5].tolist()}"
        else:
            ok = nan_a | (np.abs(a - b) <= TRAJ_ATOL + TRAJ_RTOL * np.abs(b))
            # the tolerance is a CONJUNCTION in north_star (1e-9 rel / 1e-6 m abs); report both
            err = np.where(nan_a, 0.0, np.abs(a - b))
            assert ok.all(), f"{what}{k}: max abs err {err.max():.3e} at {np.argwhere(~ok)[:5].tolist()}"
            rel = err / np.maximum(np.abs(np.where(nan_b, 1.0, b)), 1e-300)
            assert rel.max() <= TRAJ_RTOL, f"{what}{k}: max rel err {rel.max():.3e}"


def plans_dict(pb):
    return {k: getattr(pb, k) for k in pb.fields}
