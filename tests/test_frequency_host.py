"""The schedule of the mission loop (csrc/rollout_core.cuh, compiled for the host by tests/devtools/host_rollout.cpp) at outer-loop
frequencies other than 10, against the fp64 C oracle at the same frequency (main.py:37-61: outer update iff inner_step % frequency
== 0, index clamped at the last row).  rollout_run<double> carries the period phase between calls, splits the tick loop into
stretches at period boundaries, folds the position and renormalises the quaternion once per period, and counts periods for the
metrics: all of it depends on the frequency, and in fp64 it must reproduce the oracle to rounding (1e-9 m)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import rotation_angle
from oracle import c_port, flight_np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FREQS = (1, 2, 3, 7, 10, 20, 50)
TOL = 1e-9


@pytest.fixture(scope="module")
def host_rollout(tmp_path_factory):
    so = tmp_path_factory.mktemp("k2") / "libhost_rollout.so"
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", "-I", os.path.join(ROOT, "uav-autonomous-control_b200", "csrc"),
                    os.path.join(ROOT, "tests", "devtools", "host_rollout.cpp"), "-o", str(so)], check=True)
    L = ctypes.CDLL(str(so))
    dp, ip, i = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.c_int
    L.host_rollout.argtypes = [dp, ip, ip, dp, i, dp, i, i, i, i, dp, i, dp, dp, dp, dp, i, dp]
    L.host_rollout.restype = i

    def as_p(a, t):
        return None if a is None else a.ctypes.data_as(t)

    def fly(mission, start, freq, n_ticks, *, split=0, lag=1, boxes=None, goal, mc=None, log_stride=0):
        coeffs, rows, table, yaw0 = mission
        mc = np.concatenate((np.ones(15), np.zeros(3))) if mc is None else np.ascontiguousarray(mc, float)
        bx = None if boxes is None else np.ascontiguousarray(boxes, float)
        start, goal = np.ascontiguousarray(start, float), np.ascontiguousarray(goal, float)
        m, X = np.empty(8), np.empty(13)
        log = np.empty((n_ticks // log_stride, 13)) if log_stride else None
        rc = L.host_rollout(as_p(coeffs, dp), as_p(rows, ip), as_p(table, ip), as_p(yaw0, dp), len(rows), as_p(start, dp), freq, n_ticks, split,
                            lag, as_p(bx, dp), 0 if bx is None else len(bx), as_p(goal, dp), as_p(mc, dp), as_p(m, dp), as_p(X, dp), log_stride,
                            as_p(log, dp))
        assert rc == 0
        return m, X, log
    return fly


def _mission(waypoints, velocity, dt):
    """Packed segments of the take-off table + course table sampled at dt (the layout of uavb_rollout_args), and the oracle's table."""
    coeffs, rows, table, yaw0 = [], [], [], []
    for wp in (waypoints[:2], waypoints[1:]):
        c, T = c_port.solve_coeffs(wp, velocity)
        tab = c_port.sample_table(c, T, dt)
        valid = np.flatnonzero(np.hypot(tab[:, 3], tab[:, 4]) >= 1e-3)
        y0 = float(np.arctan2(tab[valid[0], 4], tab[valid[0], 3])) if len(valid) else 0.0
        for s in range(len(T)):
            coeffs.append(c[8 * s:8 * s + 8].ravel())
            rows.append(c_port.lib().oracle_sample_count(float(T[s]), float(dt)))
            table.append(1 if s == 0 else 0)
            yaw0.append(y0 if s == 0 else 0.0)
    packed = (np.ascontiguousarray(np.concatenate(coeffs)), np.array(rows, np.int32), np.array(table, np.int32), np.array(yaw0))
    return packed, c_port.mission_table(waypoints, velocity, dt)


def _compare(host, ref, what):
    m, X, _ = host
    dp = np.abs(X[:3] - ref["X"][:3]).max()
    da = float(rotation_angle(X[3:7], ref["X"][3:7]))
    assert dp < TOL and da < TOL, (what, dp, da)
    assert np.abs(X[7:] - ref["X"][7:]).max() < 1e-7, what
    assert m[7] == ref["periods"] and m[5] == 0, what
    assert m[1] == float(ref["collision"]) and m[6] == ref["first_collision_tick"], what
    for k, name in ((0, "final_dist"), (2, "rmse"), (3, "mean_err"), (4, "max_err")):
        assert abs(m[k] - ref[name]) < TOL, (what, name, m[k], ref[name])
    return dp


@pytest.mark.parametrize("freq", FREQS)
def test_mission_loop_matches_the_c_oracle_at_every_frequency(host_rollout, freq):
    g = np.load(os.path.join(ROOT, "tests", "golden", "planning.npz"))
    W, boxes = g["waypoints"], g["obstacles"]
    start, goal = W[0], W[-1]
    mission, tab = _mission(W, 3.0, 0.001 * freq)
    n_rows = len(tab)
    assert n_rows == int(mission[1].sum())
    full = freq * n_rows
    veh = flight_np.Vehicle()
    # a box on the course: the flag and the first-hit tick must be the oracle's
    mid = tab[n_rows // 2, :3]
    hit_box = np.array([[mid[0] - 0.6, mid[0] + 0.6, mid[1] - 0.6, mid[1] + 0.6, mid[2] - 0.6, mid[2] + 0.6]])
    cases = [
        ("whole mission, lab_course boxes, split inside a period", full, dict(boxes=boxes, split=(n_rows // 3) * freq + freq // 2)),
        ("box on the course", full, dict(boxes=np.vstack((boxes, hit_box)))),
        ("ticks not a multiple of the period", freq * (n_rows // 2) + freq - 1, dict(split=freq * (n_rows // 4) + 1)),
        ("fewer ticks than one period", freq - 1, dict()),
        ("past the end of the table", full + 1500 + freq // 2, dict(split=full - freq // 2)),
        ("fresh thrust frame", full, dict(lag=0)),
    ]
    worst = 0.0
    for what, n, kw in cases:
        host = host_rollout(mission, start, freq, n, goal=goal, **kw)
        ref = c_port.closed_loop(veh, tab, start, freq=freq, n_ticks=n, obstacles=kw.get("boxes"), goal=goal, thrust_frame_lag=kw.get("lag", 1))
        worst = max(worst, _compare(host, ref, what))
        if what == "box on the course":
            assert ref["collision"] and ref["first_collision_tick"] > 0
        if what == "fewer ticks than one period":
            assert host[0][7] == 0 and host[0][2] == 0 and host[0][3] == 0 and host[0][4] == 0
    # Monte-Carlo vehicle with wind, split inside a period
    rng = np.random.default_rng(freq)
    mc = np.concatenate((rng.uniform(0.9, 1.1, 4), rng.uniform(0.8, 1.2, 11), rng.uniform(-0.08, 0.08, 3)))
    d = flight_np.Vehicle()
    f = {k: getattr(d, k) for k in flight_np.Vehicle.__dataclass_fields__}
    f["mass"], f["inertia"] = d.mass * mc[0], d.inertia * mc[1:4]
    for k, name in enumerate(flight_np.Vehicle.GAIN_NAMES):
        f[name] = getattr(d, name) * mc[4 + k]
    n = full - freq // 3
    host = host_rollout(mission, start, freq, n, goal=goal, mc=mc, split=n // 2 + 1, boxes=boxes)
    ref = c_port.closed_loop(flight_np.Vehicle(**f), tab, start, freq=freq, n_ticks=n, obstacles=boxes, goal=goal, wind=mc[15:])
    worst = max(worst, _compare(host, ref, "Monte-Carlo vehicle with wind"))
    # the state once per period against the oracle's log at the same stride
    n = freq * min(n_rows, 3000)
    _, _, log = host_rollout(mission, start, freq, n, goal=goal, log_stride=freq)
    ref = c_port.closed_loop(veh, tab, start, freq=freq, n_ticks=n, goal=goal, log_stride=freq)
    assert log.shape == ref["log"].shape
    assert np.abs(log[:, :3] - ref["log"][:, :3]).max() < TOL and rotation_angle(log[:, 3:7], ref["log"][:, 3:7]).max() < TOL
    print(f"F = {freq}: {n_rows} rows, worst final-position difference {worst:.1e} m")


def test_rollout_rejects_a_plan_sampled_at_another_outer_period():
    """kernels.rollout: a MissionPlan's dt is the controller's outer dt too, so it must be vehicle.dt * frequency (main.py:97)."""
    import torch
    from uav_ac_b200 import _native as nat, kernels
    z = torch.zeros(1)
    plan = kernels.MissionPlan(z, z.int(), z.int(), z.double(), 0.01, n_seg_shared=1)
    veh = nat.Vehicle(dt=0.001, mass=0.5)
    start = torch.zeros(3, dtype=torch.float64)
    for freq in (5, 7, 11, 100):
        with pytest.raises(ValueError, match="vehicle.dt"):
            kernels.rollout(plan, 4, 100, start=start, vehicle=veh, frequency=freq)
    plan.dt = 0.001 * 7
    with pytest.raises(ValueError, match="vehicle.dt"):
        kernels.rollout(plan, 4, 100, start=start, vehicle=veh, frequency=10)
    with pytest.raises(ValueError, match="vehicle.dt"):
        kernels.rollout(plan, 4, 100, start=start, vehicle=nat.Vehicle(dt=0.002, mass=0.5), frequency=7)
    # a consistent plan gets past the check (and then needs CUDA tensors)
    with pytest.raises(nat.UavbError):
        kernels.rollout(plan, 4, 100, start=start, vehicle=veh, frequency=7)
