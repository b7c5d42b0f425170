"""Shared helpers for the parity tests (test infrastructure; may import oracle/)."""
from __future__ import annotations

import numpy as np

GOAL = np.array([23.0, 7.0, -2.0])


def normwise(c, ref):
    """Per-mission norm-wise relative error |dc|_inf / |c|_inf (SURVEY 7.3: the only meaningful 1e-9 metric)."""
    c, ref = np.asarray(c), np.asarray(ref)
    return float(np.abs(c - ref).max() / np.abs(ref).max())


def rotation_angle(qa, qb):
    """Angle of conj(qa)*qb from its vector part (well conditioned near zero); arrays [..., 4] scalar first."""
    a0, a1, a2, a3 = np.moveaxis(np.asarray(qa, float), -1, 0)
    b0, b1, b2, b3 = np.moveaxis(np.asarray(qb, float), -1, 0)
    vx = a0 * b1 - a1 * b0 - a2 * b3 + a3 * b2
    vy = a0 * b2 + a1 * b3 - a2 * b0 - a3 * b1
    vz = a0 * b3 - a1 * b2 + a2 * b1 - a3 * b0
    return 2 * np.arcsin(np.sqrt(vx * vx + vy * vy + vz * vz).clip(0, 1))


def eval_poly(coeffs, seg, t, order=0):
    """Value of derivative `order` of spline `seg` at local time t; coeffs (8S, 3) reference layout."""
    c = np.asarray(coeffs)[8 * seg:8 * seg + 8]
    out = np.zeros(c.shape[1])
    for j in range(order, 8):
        f = 1.0
        for k in range(order):
            f *= (j - k)
        out += f * c[j] * t ** (j - order)
    return out


def lab_course_plan(dev, velocity, dt=0.01):
    """MissionPlan of the lab_course mission: vertical take-off table + course table (main.py:73-84)."""
    import torch
    from uav_ac_b200 import kernels
    from uav_ac_b200.simulation.scene import LAB_COURSE_WAYPOINTS as W
    tk = torch.tensor(W[:2][None], dtype=torch.float64, device=dev)
    co = torch.tensor(W[1:][None], dtype=torch.float64, device=dev)
    vel = torch.tensor([velocity], dtype=torch.float64, device=dev)
    return kernels.plan_missions([(tk, vel), (co, vel)], dt, shared=True)


def mc_arrays(dev, B, gain_scale=None, mass_scale=None, inertia_scale=None, wind=None):
    """SoA fp32 Monte-Carlo overrides from multiplicative scales given per rollout ([B, ...] arrays)."""
    import torch
    from uav_ac_b200 import _native as nat
    v = nat.default_vehicle()
    out = {}
    if gain_scale is not None:
        g = np.asarray(list(v.gains))[None, :] * np.asarray(gain_scale, float).reshape(B, 11)
        out["mc_gains"] = torch.tensor(g.T.copy(), dtype=torch.float32, device=dev).contiguous()
    if mass_scale is not None:
        out["mc_mass"] = torch.tensor(v.mass * np.asarray(mass_scale, float).reshape(B), dtype=torch.float32, device=dev)
    if inertia_scale is not None:
        i = np.asarray(list(v.inertia))[None, :] * np.asarray(inertia_scale, float).reshape(B, 3)
        out["mc_inertia"] = torch.tensor(i.T.copy(), dtype=torch.float32, device=dev).contiguous()
    if wind is not None:
        out["mc_wind"] = torch.tensor(np.asarray(wind, float).reshape(B, 3).T.copy(), dtype=torch.float32, device=dev).contiguous()
    return out


def hover_table(start):
    """A one-row trajectory table: hold a point 0.2 m / -0.1 m off the start at 1 m altitude, yaw 0.4 rad."""
    return np.array([[start[0] + 0.2, start[1] - 0.1, -1.0, 0, 0, 0, 0, 0, 0, 0.4, 0]])


def rough_mc(dev, B, seed=11, tumble=False):
    """Wind +-0.3 N and gains x U(0.5, 1.5) (most stretches of a warp see some lane at a rotor limit); tumble: every other rollout is a
    low-inertia vehicle with four times the attitude gains (with a yaw set-point 3 rad away, |w| goes well above 44.7 rad/s)."""
    rng = np.random.default_rng(seed)
    gains = rng.uniform(0.5, 1.5, (B, 11))
    inertia = np.ones((B, 3))
    if tumble:
        gains[::2] = 1.0
        gains[::2, [5, 6, 8, 9]] = 4.0
        inertia[::2] = 0.1
    return mc_arrays(dev, B, gain_scale=gains, inertia_scale=inertia, wind=rng.uniform(-0.3, 0.3, (B, 3)))
