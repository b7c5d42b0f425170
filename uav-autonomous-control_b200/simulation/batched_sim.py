"""``BatchedSimulation``: the stand-in for ``MujocoSimulation`` (``uav_ac/simulation/mujoco_sim.py:48-347``)
on the batched path.  MuJoCo is never involved: the single free-joint body that ``mj_step`` integrates
is restated as the semi-implicit Euler step of SURVEY 8(a) D2 inside the CUDA kernels, and contacts are
replaced by the inclusive point-in-AABB flag of ``minimum_snap.py:327-357`` (BASELINE.json north_star).

Two ways to advance the drones:

* ``step()`` -- one 1 kHz tick for all B drones, after ``trajectory_controller.step()``, exactly like the
  headless loop of ``tests/integration/test_mujoco_trajectory_tracking.py:27-31`` (method-level parity;
  one kernel launch per call);
* ``rollout()`` -- the whole mission in ONE persistent kernel launch (K2), state in registers.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from .. import _native as nat, _stages as st, kernels
from ..quadrotor.quad import Quad
from . import scene


class BatchedSimulation:
    TAKEOFF_HEIGHT = 0.1   # mujoco_sim.py:17 (ground-contact amnesty; unused by the free-body model)
    ACTUAL_TRAJECTORY_SAMPLE_INTERVAL = 0.05   # mujoco_sim.py:16
    ACTUAL_TRAJECTORY_SEGMENT_COUNT = 200      # mujoco_sim.py:14 (capsules the viewer can draw; the list itself is unbounded)

    def __init__(self, batch: int = 1, device=None, *, model_path=None, waypoints=None, obstacles=None, thrust_frame_lag: int = 1,
                 mass=None, inertia=None):
        """lab_course scene by default (constants transcribed from lab_course.xml, ``simulation/scene.py``); ``model_path``
        reads any MJCF scene of the same conventions with the stdlib reader (``scene.load_scene``; the reference passes
        the path to ``MujocoSimulation(model_path)``, mujoco_sim.py:51).
        ``thrust_frame_lag=1`` reproduces the headless loop (stale ``data.xmat``), 0 the viewer callback path."""
        self.batch = int(batch)
        self._scene = scene.load_scene(model_path) if model_path is not None else None
        if self._scene is not None:
            waypoints = self._scene.mission_waypoints if waypoints is None else waypoints
            obstacles = self._scene.obstacles if obstacles is None else obstacles
        self.mission_waypoints = np.array(scene.LAB_COURSE_WAYPOINTS if waypoints is None else waypoints, dtype=float)
        self.obstacles = np.array(scene.LAB_COURSE_OBSTACLES if obstacles is None else obstacles, dtype=float).reshape(-1, 6)
        self.goal_position = self.mission_waypoints[-1].copy()
        self.thrust_frame_lag = int(thrust_frame_lag)
        self.quad = self._create_quad(device, mass, inertia)
        self.device = self.quad.device
        self._obs = torch.tensor(self.obstacles, dtype=torch.float32, device=self.device)
        self.wind = None           # optional (B, 3) constant force in N (extension; BASELINE configs[3])
        self._reset_runtime_state()
        for box in self.obstacles:     # mujoco_sim.py:90-91
            s = self.mission_waypoints[0]
            if box[0] <= s[0] <= box[1] and box[2] <= s[1] <= box[3] and box[4] <= s[2] <= box[5]:
                raise ValueError("the start position is inside an obstacle")

    def _create_quad(self, device, mass, inertia) -> Quad:
        """Arguments of ``_create_quad`` for lab_course.xml (mujoco_sim.py:258-279)."""
        if self._scene is not None:
            kw = self._scene.quad_kwargs()
            if mass is not None:
                kw["mass"] = mass
            if inertia is not None:
                kw["inertia"] = inertia
            return Quad(batch=self.batch, device=device, **kw)
        d = nat.default_vehicle()
        return Quad(g=d.g, dt=d.dt, mass=d.mass if mass is None else mass, inertia=list(d.inertia) if inertia is None else inertia,
                    arm_length=d.arm, force_coefficient=d.kf, drag_to_thrust=d.kappa, thrust_limits=[d.min_thrust, d.max_thrust],
                    motor_time_constants=[d.tau_rise, d.tau_fall],
                    flight_limits=[d.max_ascent, d.max_descent, d.max_speed_xy, d.max_horiz_accel, d.max_tilt], batch=self.batch, device=device)

    def _reset_runtime_state(self) -> None:
        """Back to the start pose with rotors at rest (mujoco_sim.py:190-199)."""
        q = self.quad
        q.X.zero_()
        q.X[:, 0:3] = torch.tensor(self.mission_waypoints[0], dtype=torch.float32, device=self.device)
        q.X[:, 3] = 1.0
        q.omega.zero_()
        q.omega_command.zero_()
        self._collided = torch.zeros((self.batch,), dtype=torch.float32, device=self.device)
        self._zb = torch.zeros((3, self.batch), dtype=torch.float32, device=self.device)
        self._zb[2] = 1.0          # body z axis of the identity attitude (mj_forward in __init__, mujoco_sim.py:81)
        self.time = 0.0

    @property
    def collision_detected(self) -> torch.Tensor:
        """(B,) bool, sticky (mujoco_sim.py:93-101; AABB semantics on the batched path)."""
        return self._collided > 0

    has_collision = collision_detected

    def step(self) -> torch.Tensor:
        """One physics tick for every drone (mujoco_sim.py:144-151): rotor wrench with the stale (or fresh) thrust
        frame, free-body step, state sync, collision bookkeeping.  Returns a copy of ``quad.X``."""
        q = self.quad
        B = self.batch
        X = st.soa(q.X)
        zb_next = torch.empty_like(self._zb)
        st.run(nat.STAGE_PHYSICS, q, q.dt, B, X=X, omega=st.soa(q.omega), zb=self._zb if self.thrust_frame_lag else None,
               zb_out=zb_next, wind=st.soa(self.wind) if self.wind is not None else None,
               aabbs=self._obs if len(self.obstacles) else None, n_obs=len(self.obstacles), collided=self._collided)
        self._zb = zb_next
        q.X = X.t().contiguous()
        self.time += q.dt
        return q.X.clone()

    # ------------------------------------------------------------------ fused path
    def rollout(self, velocity: float, frequency: int = 10, n_ticks: Optional[int] = None, *, gains: Optional[dict] = None,
                log_stride: int = 0, want_state: bool = True, record_actual_trajectory: bool = False, ground: bool = False):
        """Plan the mission (take-off table + course table, each with the obstacle-correction loop, main.py:73-84) and fly it for every drone in one launch of
        the persistent rollout kernel.  ``gains`` maps gain names to (B,) tensors (Monte-Carlo); mass / inertia
        perturbations come from the Quad.  Returns ``kernels.RolloutResult`` (metrics (B, 8), final state, log).
        ``record_actual_trajectory``: also keep every drone's flown-path list exactly as the viewer records it
        (``_record_actual_trajectory``, mujoco_sim.py:201-218: one position per 0.05 s of simulation time while the drone is at or
        above the take-off altitude ``mission_waypoints[1][2]``) in ``result.traj`` / ``result.traj_count``.
        ``ground``: unilateral floor at the start height (the reference's drone rests on MuJoCo's ground plane until its rotors
        carry it; the default free body sags ~1.5 cm through it in the first 50 ms, SURVEY 7.3)."""
        q = self.quad
        dev = self.device
        wp = torch.tensor(self.mission_waypoints, dtype=torch.float64, device=dev)
        vel = torch.tensor([float(velocity)], dtype=torch.float64, device=dev)
        obs64 = torch.tensor(self.obstacles, dtype=torch.float64, device=dev) if len(self.obstacles) else None
        plan = kernels.plan_missions([(wp[None, :2].contiguous(), vel), (wp[None, 1:].contiguous(), vel)], q.dt * frequency, shared=True,
                                     obstacles=obs64)       # both tables through the correction loop, like _generate_mission_trajectory
        if n_ticks is None:
            n_ticks = frequency * int(plan.total_rows.item())
        veh, mc = q.vehicle_struct(self.batch, gains or {})
        return kernels.rollout(plan, self.batch, n_ticks, start=wp[0].contiguous(), goal=wp[-1].contiguous(), vehicle=veh, frequency=frequency,
                               mc_mass=mc.get("mc_mass"), mc_inertia=mc.get("mc_inertia"), mc_gains=mc.get("mc_gains"),
                               mc_wind=st.soa(self.wind) if self.wind is not None else None,
                               obstacles=self._obs if len(self.obstacles) else None, thrust_frame_lag=self.thrust_frame_lag,
                               log_stride=log_stride, want_state=want_state, ground_z=float(self.mission_waypoints[0][2]) if ground else None,
                               traj_max_samples=(n_ticks // int(round(self.ACTUAL_TRAJECTORY_SAMPLE_INTERVAL / q.dt)) + 1) if record_actual_trajectory else 0,
                               traj_gate_z=float(self.mission_waypoints[1][2]), traj_interval=self.ACTUAL_TRAJECTORY_SAMPLE_INTERVAL)

    def fly_trajectory(self, trajectory, frequency: int = 10, n_ticks: Optional[int] = None, *, table_index=None, start=None, goal=None,
                       gains: Optional[dict] = None, log_stride: int = 0, want_state: bool = True, record_actual_trajectory: bool = False,
                       ground: bool = False):
        """Fly caller-supplied (N, 11) trajectory tables [x y z vx vy vz ax ay az yaw spline_id] in one launch of the persistent
        rollout kernel: ``TrajectoryController(controller, quad, trajectory, frequency)`` followed by ``step()`` over the table
        (main.py:10-61) for every drone -- one row per ``frequency`` ticks, the index held at the last row.

        ``trajectory``: one table flown by every drone, a (T, N, 11) stack or a sequence of (N_t, 11) tables with ``table_index``
        (B,) choosing each drone's table (None: drone b flies table b), or a ``kernels.TablePlan``.  ``start``: [3] or (B, 3), default
        the scene start; ``goal`` (for final_dist): default the last row's position of each drone's table; ``n_ticks``: default
        ``frequency`` x the rows of the longest table.  Mass / inertia, ``gains`` and ``self.wind`` as in ``rollout()``.
        Returns ``kernels.RolloutResult``."""
        q = self.quad
        dev = self.device
        if isinstance(trajectory, kernels.TablePlan):
            if table_index is not None:
                raise ValueError("table_index belongs to the TablePlan (kernels.plan_tables)")
            plan = trajectory
        else:
            plan = kernels.plan_tables(trajectory, table_index, device=dev)
        if n_ticks is None:
            n_ticks = frequency * plan.max_rows
        start = torch.tensor(self.mission_waypoints[0], dtype=torch.float64, device=dev) if start is None else \
            torch.as_tensor(start, dtype=torch.float64).to(dev).contiguous()
        goal = plan.goals(self.batch) if goal is None else torch.as_tensor(goal, dtype=torch.float64).to(dev).contiguous()
        veh, mc = q.vehicle_struct(self.batch, gains or {})
        return kernels.rollout(plan, self.batch, n_ticks, start=start, goal=goal, vehicle=veh, frequency=frequency,
                               mc_mass=mc.get("mc_mass"), mc_inertia=mc.get("mc_inertia"), mc_gains=mc.get("mc_gains"),
                               mc_wind=st.soa(self.wind) if self.wind is not None else None,
                               obstacles=self._obs if len(self.obstacles) else None, thrust_frame_lag=self.thrust_frame_lag,
                               log_stride=log_stride, want_state=want_state, ground_z=float(self.mission_waypoints[0][2]) if ground else None,
                               traj_max_samples=(n_ticks // int(round(self.ACTUAL_TRAJECTORY_SAMPLE_INTERVAL / q.dt)) + 1) if record_actual_trajectory else 0,
                               traj_gate_z=float(self.mission_waypoints[1][2]), traj_interval=self.ACTUAL_TRAJECTORY_SAMPLE_INTERVAL)
