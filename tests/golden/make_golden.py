#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REFERENCE's own classes in the build container.

Run from the repo root (needs /root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

Everything on the path is executed by the reference objects -- ``MinimumSnap``,
``CascadedController``, ``Quad``, ``TrajectoryController``, ``_generate_mission_trajectory`` --
imported from /root/reference with a stub ``mujoco`` module (SURVEY appendix B).  The one piece the
reference does not own, the MuJoCo rigid-body step, is replaced by ``oracle.freebody.freebody_step``
(parity unpinned at that boundary; see its header).  The committed .npz files are what the oracle
(tests -m "not gpu") and the CUDA path (tests -m gpu) are compared with.
"""
from __future__ import annotations

import os
import sys
import unittest.mock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")
sys.modules["mujoco"] = unittest.mock.MagicMock()

from uav_ac.control.controller import CascadedController  # noqa: E402
from uav_ac.main import TrajectoryController, _generate_mission_trajectory  # noqa: E402
from uav_ac.planning.minimum_snap import MinimumSnap  # noqa: E402
from uav_ac.quadrotor.quad import Quad  # noqa: E402

from oracle.freebody import freebody_step  # noqa: E402

# lab_course scene, NED (reference tests/unit/simulation/test_mujoco_sim.py:40-50, :246; SURVEY 8(a) P9)
WAYPOINTS = np.array([[1, 7, -0.021], [1, 7, -1.3], [4, 7, -1.3], [7.5, 4, -3], [11, 7, -3.5], [14, 10, -2.5],
                      [17, 10, -3.2], [20.5, 7, -1.4], [23, 7, -2]], dtype=float)
OBSTACLES = np.array([[3.7, 4.3, 4, 10, -3.4, -2.8], [10.7, 11.3, 4, 10, -2.2, 0], [13.3, 14.7, 6.3, 7.7, -6, 0],
                      [20.2, 20.8, 4, 10, -3.3, -2.7]], dtype=float)
GOAL = np.array([23.0, 7.0, -2.0])
FREQ = 10
GAIN_NAMES = ("kp_xy", "kd_xy", "kp_z", "kd_z", "ki_z", "kp_roll", "kp_pitch", "kp_yaw", "kp_p", "kp_q", "kp_r")


def make_quad() -> Quad:
    """Arguments of mujoco_sim._create_quad for lab_course.xml (SURVEY 3.1)."""
    return Quad(g=9.81, dt=0.001, mass=0.5, inertia=np.array([0.0023, 0.0023, 0.0046]), arm_length=0.120208,
                force_coefficient=1.0, drag_to_thrust=0.016, thrust_limits=np.array([0.1, 4.5]),
                motor_time_constants=np.array([0.0125, 0.025]), flight_limits=np.array([3.0, 2.0, 3.0, 12.0, 0.7]))


def c2_missions(rng, n, S=4):
    """BASELINE configs[1] generator (SURVEY 8(d) C2): bounded-duration random missions."""
    w = np.empty((n, S + 1, 3))
    w[:, 0] = rng.uniform([2, 2, -5], [22, 12, -1], size=(n, 3))
    for i in range(S):
        u = rng.normal(size=(n, 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        u[:, 2] *= 0.4
        step = rng.uniform(2.0, 5.0, size=(n, 1))
        w[:, i + 1] = w[:, i] + step * u
    vel = rng.uniform(2.0, 3.0, size=n)
    return w, vel


def planning():
    out = {"waypoints": WAYPOINTS, "obstacles": OBSTACLES}
    ks, ts = np.arange(7), np.array([0.0, 3.0, 0.37, 1.9])
    out["polynom_t"] = ts
    out["polynom"] = np.array([[MinimumSnap.polynom(8, int(k), float(t)) for t in ts] for k in ks])
    for v in (2.0, 3.0):
        tag = f"v{int(v)}"
        for name, wp in (("takeoff", WAYPOINTS[:2]), ("course", WAYPOINTS[1:])):
            for method in ("lstsq", "solve"):
                ms = MinimumSnap(wp, None, v, 0.01)
                ms._compute_spline_parameters(method)
                out[f"{tag}_{name}_coeffs_{method}"] = np.asarray(ms.coeffs)
            out[f"{tag}_{name}_times"] = np.asarray(ms.times)
            out[f"{tag}_{name}_A"] = ms.A
            out[f"{tag}_{name}_b"] = ms.b
            out[f"{tag}_{name}_Q"] = ms._create_snap_cost_matrix()
        out[f"{tag}_table"] = _generate_mission_trajectory(WAYPOINTS, OBSTACLES, v, 0.01)
    # random bounded missions, S=4 (C2) and ragged S
    rng = np.random.default_rng(20261017)
    w, vel = c2_missions(rng, 64, 4)
    cs, cl, tt = [], [], []
    for i in range(len(w)):
        ms = MinimumSnap(w[i], None, float(vel[i]), 0.01)
        ms._compute_spline_parameters("solve")
        cs.append(np.asarray(ms.coeffs))
        tt.append(np.asarray(ms.times))
        ms = MinimumSnap(w[i], None, float(vel[i]), 0.01)
        ms._compute_spline_parameters("lstsq")
        cl.append(np.asarray(ms.coeffs))
    out.update(c2_waypoints=w, c2_velocity=vel, c2_coeffs_solve=np.array(cs), c2_coeffs_lstsq=np.array(cl), c2_times=np.array(tt))
    for S in (1, 2, 3, 5, 8, 12):
        w, vel = c2_missions(rng, 6, S)
        cs, tt = [], []
        for i in range(len(w)):
            ms = MinimumSnap(w[i], None, float(vel[i]), 0.01)
            ms._compute_spline_parameters("solve")
            cs.append(np.asarray(ms.coeffs))
            tt.append(np.asarray(ms.times))
        out[f"rag{S}_waypoints"], out[f"rag{S}_velocity"] = w, vel
        out[f"rag{S}_coeffs_solve"], out[f"rag{S}_times"] = np.array(cs), np.array(tt)
    # one sampled table of a random mission (no obstacles) for the sampler / yaw rows
    ms = MinimumSnap(out["c2_waypoints"][3], None, float(out["c2_velocity"][3]), 0.01)
    out["c2_table3"] = ms.get_trajectory()
    # yaw profiles (ms:126-136)
    yv, yy = [], []
    for case in range(6):
        n = 40
        v = rng.normal(size=(n, 3)) * (1.0 if case < 4 else 1e-4)
        if case == 1:
            v[:7, :2] = 1e-5            # invalid head: look-ahead to the first valid row
        if case == 2:
            ang = np.linspace(0, 4 * np.pi, n)  # two full turns: unwrap
            v[:, 0], v[:, 1] = np.cos(ang), np.sin(ang)
            v[10:14, :2] *= 1e-6
        if case == 3:
            v[20:, :2] = 0.0
        yv.append(v)
        yy.append(MinimumSnap._calculate_yaws(v))
    out["yaw_vel"], out["yaw_out"] = np.array(yv), np.array(yy)
    # collision truth table and midpoint insertion (reference tests :7-19, :186-200)
    box = np.array([0.0, 1.0, -1.0, 2.0, 3.0, 4.0])
    pts = np.array([[0, -1, 3], [1, 2, 4], [0.5, 0.5, 3.5], [-1e-12, 0, 3.5], [0.5, 2.0000001, 3.5], [0.5, 0, 4.1], [1, -1, 4]], dtype=float)
    out["aabb_box"], out["aabb_pts"] = box, pts
    out["aabb_hit"] = np.array([MinimumSnap.is_collision_cuboid(*p, box) for p in pts])
    p5 = rng.normal(size=(5, 3))
    out["mid_points"] = p5
    out["mid_out_13"] = MinimumSnap.insert_midpoints_at_indexes(p5, [1, 3])
    out["mid_out_2"] = MinimumSnap.insert_midpoints_at_indexes(p5, {2})
    # obstacle-driven midpoint insertion (reference test :171-183 style: obstacles where the unconstrained spline bulges)
    wp = np.array([[0.0, 0.0, -1.0], [4.0, 0.0, -1.0], [4.0, 4.0, -1.0], [8.0, 4.0, -1.5]])
    obs = np.array([[4.1, 4.6, 0.5, 1.2, -1.2, -0.8], [2.0, 2.7, -0.6, -0.35, -1.2, -0.8]])
    ms = MinimumSnap(wp, obs, 1.5, 0.01)
    tab = ms.get_trajectory()
    out.update(fix_waypoints_in=wp, fix_obstacles=obs, fix_waypoints_out=np.asarray(ms.waypoints), fix_table=tab,
               fix_coeffs=np.asarray(ms.coeffs), fix_times=np.asarray(ms.times))
    np.savez_compressed(os.path.join(HERE, "planning.npz"), **out)
    print("planning.npz:", {k: np.asarray(v).shape for k, v in out.items() if k.endswith("table") or k.startswith("fix_w")})


def stages():
    """Random inputs through the reference's stage methods (ctl:26-168, quad:88-122)."""
    rng = np.random.default_rng(7)
    n = 96
    quad = make_quad()
    out = {}
    # random attitudes up to ~35 deg tilt
    ax = rng.normal(size=(n, 3))
    ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    ang = rng.uniform(-0.6, 0.6, size=n)
    quat = np.concatenate((np.cos(ang / 2)[:, None], np.sin(ang / 2)[:, None] * ax), axis=1)
    quat[:8] *= rng.uniform(0.9, 1.1, size=(8, 1))  # un-normalised on purpose (quad:141 normalises, :190-213 do not)
    X = np.zeros((n, 13))
    X[:, 0:3] = rng.uniform([0, 0, -6], [24, 14, 0], size=(n, 3))
    X[:, 3:7] = quat
    X[:, 7:10] = rng.normal(size=(n, 3)) * 2
    X[:, 10:13] = rng.normal(size=(n, 3)) * 1.5
    des = rng.normal(size=(n, 3, 3)) * np.array([3.0, 3.0, 4.0])  # [axis][pos, vel, acc]
    des[:, :, 0] += X[:, 0:3]
    psi_des = rng.uniform(-8, 8, size=n)
    integ0 = rng.uniform(-10.5, 10.5, size=n)
    thrust, integ1, bxy, pq, rc, Rm, eul = [], [], [], [], [], [], []
    for i in range(n):
        quad.X = X[i].copy()
        ctrl = CascadedController(9.81, 0.01)
        ctrl.integral_error = integ0[i]
        R = quad.R()
        c = ctrl.altitude(quad, des[i, 2], R, quad.kp_z, quad.kd_z, quad.ki_z)
        b = ctrl.lateral(quad, des[i, 0], des[i, 1], c, quad.kp_xy, quad.kd_xy)
        pqc = ctrl.roll_pitch_controller(b, R, quad.kp_roll, quad.kp_pitch)
        r = ctrl.yaw_controller(quad, psi_des[i], quad.kp_yaw, pqc[1])
        thrust.append(c); integ1.append(ctrl.integral_error); bxy.append(b); pq.append(pqc); rc.append(r)
        Rm.append(R); eul.append(quad.euler_angles)
    out.update(X=X, des=des, psi_des=psi_des, integ0=integ0, thrust=np.array(thrust), integ1=np.array(integ1),
               bxy=np.array(bxy), pq=np.array(pq), r_c=np.array(rc), R=np.array(Rm), euler=np.array(eul))
    # body-rate loop, allocation and motor lag incl. saturating cases
    pqr_cmd = rng.normal(size=(n, 3)) * 3
    tcmd = rng.uniform(-1, 20, size=n)
    mom, forces, om0, om1, omc = [], [], [], [], []
    ctrl = CascadedController(9.81, 0.01)
    for i in range(n):
        quad.X = X[i].copy()
        m = ctrl.body_rate_controller(quad, pqr_cmd[i], quad.kp_p, quad.kp_q, quad.kp_r)
        if i % 3 == 0:
            m = m * 0.02                      # unsaturated cases
        f = quad._allocate_rotor_forces(tcmd[i], m)
        quad.omega = rng.uniform(0, 2.2, size=4)
        om0.append(quad.omega.copy())
        quad.set_propeller_speed(tcmd[i], m)
        mom.append(m); forces.append(f); om1.append(quad.omega.copy()); omc.append(quad.omega_command.copy())
    out.update(pqr_cmd=pqr_cmd, thrust_cmd=tcmd, moment=np.array(mom), forces=np.array(forces), omega0=np.array(om0),
               omega1=np.array(om1), omega_cmd=np.array(omc))
    ang = np.array([0.0, np.pi, -np.pi, 3 * np.pi, -3 * np.pi, 7.0, -7.0, 1e-9, 2 * np.pi, -2 * np.pi, 12.56])
    out.update(wrap_in=ang, wrap_pi=np.array([CascadedController.wrap_to_pi(a) for a in ang]),
               wrap_2pi=np.array([CascadedController.wrap_to_2pi(a) for a in ang]))
    q = make_quad()
    out["gains"] = np.array([getattr(q, g) for g in GAIN_NAMES])
    np.savez_compressed(os.path.join(HERE, "stages.npz"), **out)
    print("stages.npz written")


def fly(table, start, *, gain_scale=None, mass_scale=1.0, inertia_scale=None, wind=None, lag=1, obstacles=OBSTACLES,
        goal=GOAL, full_rate_ticks=2000):
    """Loop of the reference integration test (:26-31) with simulation.step() -> freebody_step."""
    quad = make_quad()
    if gain_scale is not None:
        for g, s in zip(GAIN_NAMES, gain_scale):
            setattr(quad, g, getattr(quad, g) * float(s))
    quad.m *= mass_scale
    if inertia_scale is not None:
        quad.i_x, quad.i_y, quad.i_z = quad.i_x * inertia_scale[0], quad.i_y * inertia_scale[1], quad.i_z * inertia_scale[2]
    quad.X[0:3] = start
    ctrl = CascadedController(quad.g, quad.dt * FREQ)
    tc = TrajectoryController(ctrl, quad, table, FREQ)
    R_stale = quad.R()
    Xs, oms, integ, errs, fine, thr = [], [], [], [], [], []
    collided, first_hit, k = False, -1, 0
    for target in table:
        for _ in range(FREQ):
            tc.step()
            R_now = quad.R()
            quad.X = freebody_step(quad.X, quad.omega, R_stale if lag else R_now, g=quad.g, dt=quad.dt, mass=quad.m,
                                   inertia=np.array([quad.i_x, quad.i_y, quad.i_z]), kf=quad.kf, arm=quad.l,
                                   kappa=quad.kappa, wind=wind)
            R_stale = R_now
            if not collided and obstacles is not None:
                for box in obstacles:
                    if MinimumSnap.is_collision_cuboid(*quad.position, box):
                        collided, first_hit = True, k
                        break
            if k < full_rate_ticks:
                fine.append(np.concatenate((quad.X, quad.omega)))
            k += 1
        Xs.append(quad.X.copy()); oms.append(quad.omega.copy()); integ.append(float(ctrl.integral_error))
        thr.append(np.concatenate(([tc.thrust_cmd], tc.pqr_cmd)))
        errs.append(np.linalg.norm(quad.position - target[:3]))
    errs = np.array(errs)
    return dict(X=np.array(Xs), omega=np.array(oms), integral=np.array(integ), errors=errs, cmd=np.array(thr),
                fine=np.array(fine), collision=np.array(collided), first_collision_tick=np.array(first_hit),
                final_dist=np.array(np.linalg.norm(quad.position - goal)), mean_err=np.array(errs.mean()),
                rmse=np.array(np.sqrt(np.mean(errs ** 2))), max_err=np.array(errs.max()))


def closed_loops():
    for v in (2.0, 3.0):
        table = _generate_mission_trajectory(WAYPOINTS, OBSTACLES, v, 0.01)
        res = fly(table, WAYPOINTS[0])
        np.savez_compressed(os.path.join(HERE, f"closed_loop_v{int(v)}.npz"), velocity=np.array(v), **res)
        print(f"closed_loop_v{int(v)}: rows {len(table)} final {float(res['final_dist']):.5f} mean {float(res['mean_err']):.5f} "
              f"max {float(res['max_err']):.4f} collision {bool(res['collision'])}")
    # variants on the v=3 mission: thrust-frame lag off; Monte-Carlo gains/mass/inertia; wind; an obstacle on the path
    table = _generate_mission_trajectory(WAYPOINTS, OBSTACLES, 3.0, 0.01)
    rng = np.random.default_rng(99)
    var = {}
    unused = ("fine", "cmd")                      # no test reads them for the variants; left out to keep the file under 1 MB
    res = fly(table, WAYPOINTS[0], lag=0, full_rate_ticks=0)
    var.update({f"nolag_{k}": v for k, v in res.items() if k not in unused})
    for j in range(3):
        gs, m, ins = rng.uniform(0.8, 1.2, 11), float(rng.uniform(0.9, 1.1)), rng.uniform(0.9, 1.1, 3)
        res = fly(table, WAYPOINTS[0], gain_scale=gs, mass_scale=m, inertia_scale=ins, full_rate_ticks=0)
        var.update({f"mc{j}_{k}": v for k, v in res.items() if k not in unused})
        var[f"mc{j}_gain_scale"], var[f"mc{j}_mass_scale"], var[f"mc{j}_inertia_scale"] = gs, np.array(m), ins
    wind = np.array([0.10, -0.06, 0.04])
    res = fly(table, WAYPOINTS[0], wind=wind, full_rate_ticks=0)
    var.update({f"wind_{k}": v for k, v in res.items() if k not in unused})
    var["wind_force"] = wind
    blocker = np.vstack((OBSTACLES, [[8.0, 9.0, 3.0, 6.0, -4.0, -2.0]]))  # sits on the course: the flag must trip
    res = fly(table, WAYPOINTS[0], obstacles=blocker, full_rate_ticks=0)
    var.update({f"hit_{k}": v for k, v in res.items() if k not in unused})
    var["hit_obstacles"] = blocker
    np.savez_compressed(os.path.join(HERE, "closed_loop_variants.npz"), **var)
    print("variants:", {k: float(v) for k, v in var.items() if k.endswith("final_dist") or k.endswith("first_collision_tick")})


def actual_trajectory():
    """D5: the 20 Hz position list of the viewer (mujoco_sim.py:201-218), produced by the reference's OWN
    MujocoSimulation._record_actual_trajectory running on a stand-in object (MuJoCo itself is absent): after every tick the
    simulation time advances by dt (mj_step) and the method decides -- take-off gate on quad.z, then one sample per
    ACTUAL_TRAJECTORY_SAMPLE_INTERVAL -- whether quad.position is appended.  Stored: the ticks after which a sample was taken, the
    sampled positions, and the full-rate position log they were taken from."""
    import types
    from uav_ac.simulation import mujoco_sim as ms
    table = _generate_mission_trajectory(WAYPOINTS, OBSTACLES, 3.0, 0.01)
    quad = make_quad()
    quad.X[0:3] = WAYPOINTS[0]
    ctrl = CascadedController(quad.g, quad.dt * FREQ)
    tc = TrajectoryController(ctrl, quad, table, FREQ)
    sim = types.SimpleNamespace(mission_waypoints=WAYPOINTS, quad=quad, data=types.SimpleNamespace(time=0.0),
                                _next_actual_trajectory_sample_time=0.0, _actual_trajectory_positions=[],
                                _actual_trajectory_segment_ids=None, _set_trajectory_segments=lambda *a, **k: None)
    R_stale = quad.R()
    ticks, log = [], []
    for k in range(FREQ * len(table)):
        tc.step()
        R_now = quad.R()
        quad.X = freebody_step(quad.X, quad.omega, R_stale, g=quad.g, dt=quad.dt, mass=quad.m, inertia=np.array([quad.i_x, quad.i_y, quad.i_z]),
                               kf=quad.kf, arm=quad.l, kappa=quad.kappa)
        R_stale = R_now
        sim.data.time += quad.dt                                  # mj_step advances data.time by the model time step
        before = len(sim._actual_trajectory_positions)
        ms.MujocoSimulation._record_actual_trajectory(sim)
        if len(sim._actual_trajectory_positions) > before:
            ticks.append(k)
        log.append(quad.position.copy())
    np.savez_compressed(os.path.join(HERE, "actual_trajectory.npz"), ticks=np.array(ticks), positions=np.array(sim._actual_trajectory_positions),
                        log=np.array(log), interval=np.array(ms.ACTUAL_TRAJECTORY_SAMPLE_INTERVAL), takeoff_z=np.array(WAYPOINTS[1][2]))
    print("actual_trajectory.npz:", len(ticks), "samples, first after tick", ticks[0], "spacing", sorted(set(np.diff(ticks).tolist())))


def rrt():
    """Reference RRTStar (uav_ac/planning/rrt.py) fed with the Philox stream of oracle/rrt_np.py (the stream the CUDA kernel draws
    from) through a patched np.random.uniform: best paths, their greedy simplification, slab-test truth table."""
    import contextlib
    import io
    from uav_ac.planning.rrt import RRTStar
    from oracle import rrt_np

    def run_ref(limits, start, goal, step, iters, obs, seed, mission):
        state = {"it": -1, "k": 0, "u": None}

        def fake_uniform(lo, hi):       # the reference draws uniform(0, 1) and, unless it samples the goal, three uniform(lo, hi)
            if lo == 0 and hi == 1 and state["k"] == 0:
                state["it"] += 1
                state["u"] = rrt_np.philox_u01(seed, mission, state["it"])
                state["k"] = 1 if state["u"][0] >= 0.15 else 0
                return state["u"][0]
            k = state["k"]
            state["k"] = (k + 1) % 4
            return lo + (hi - lo) * state["u"][k]

        r = RRTStar(limits, start, goal, step, iters, obs)
        with unittest.mock.patch("numpy.random.uniform", fake_uniform), contextlib.redirect_stdout(io.StringIO()):
            r.run()
        return r

    limits = np.array([[0, 0, -6.0], [24, 14, 0]])
    out = {"limits": limits, "obstacles": OBSTACLES, "step": np.array(1.5), "iters": np.array(1500), "seed": np.array(20261017)}
    starts = np.array([[1, 7, -1.3], [2, 2, -1.0], [22, 12, -4.0], [1, 13, -5.0], [12, 1, -0.5], [3, 7, -3.1]])
    goals = np.array([[23, 7, -2.0], [22, 12, -3.0], [2, 3, -1.5], [23, 1, -1.0], [12, 13, -5.5], [5, 7, -3.1]])
    out["starts"], out["goals"] = starts, goals
    for m in range(len(starts)):
        r = run_ref(limits, starts[m], goals[m], 1.5, 1500, OBSTACLES, 20261017, m)
        out[f"path{m}"] = r.best_path
        out[f"simple{m}"] = r.simplify_path(r.best_path)
        out[f"cost{m}"] = np.array(RRTStar.path_cost(r.best_path))
    r = run_ref(limits, starts[0], goals[0], 1.5, 1500, None, 20261017, 0)          # no obstacles
    out["path_free"] = r.best_path
    rng = np.random.default_rng(3)
    p, q = rng.uniform([0, 0, -6], [24, 14, 0], (400, 3)), rng.uniform([0, 0, -6], [24, 14, 0], (400, 3))
    q[:40] = p[:40] + rng.normal(size=(40, 3)) * [1.0, 0, 0]                        # axis-parallel segments (|d| < 1e-12 branches)
    hits = np.array([[RRTStar._segment_intersects_cuboid(p[i], q[i], box) for box in OBSTACLES] for i in range(len(p))])
    out.update(seg_p=p, seg_q=q, seg_hits=hits)
    np.savez_compressed(os.path.join(HERE, "rrt.npz"), **out)
    print("rrt.npz:", {k: v.shape for k, v in out.items() if k.startswith("path")}, "segment hits", int(hits.any(axis=1).sum()), "of", len(p))


def scene():
    """The reference's lab_course.xml, copied as is: tests/test_scene_reader.py checks the transcribed scene constants against it."""
    import shutil
    import uav_ac
    shutil.copyfile(os.path.join(os.path.dirname(uav_ac.__file__), "simulation", "models", "lab_course.xml"), os.path.join(HERE, "lab_course.xml"))


if __name__ == "__main__":
    which = sys.argv[1:] or ["planning", "stages", "closed_loops", "actual_trajectory", "rrt", "scene"]
    for w in which:
        globals()[w]()
