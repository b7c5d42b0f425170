"""Caller-supplied (N, 11) trajectory tables in the persistent rollout kernel (uavb_table_targets_f64, uavb_rollout_tables_f32,
kernels.plan_tables, BatchedSimulation.fly_trajectory): the seam TrajectoryController(controller, quad, trajectory, frequency) of
main.py:10-61 for a whole batch, one shared table or one table per rollout.

Anchors: the reference's own closed loop on its own table (tests/golden/closed_loop_v3.npz), the fp64 C oracle
(oracle/c_port.closed_loop) on tables that are not minimum-snap output, the NumPy oracle for the flown-path list.  Budget as for the
waypoint rollouts: 1e-4 m / 1e-4 rad; collision flags and first-hit ticks exact outside the 1e-4 m band around a box face."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import GOAL, rotation_angle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POS_TOL, ANG_TOL = 1e-4, 1e-4
FREQ, DT = 10, 0.001
START = np.array([1.0, 7.0, -0.021])            # lab_course start (LAB_COURSE_WAYPOINTS[0])


# ------------------------------------------------------------------------------------------ tables that are not min-snap output
def circle_table(n=2000, r=2.0, turns_yaw=3.0):
    """A climbing circle whose yaw column climbs through `turns_yaw` full turns (values far outside +-pi)."""
    t = np.arange(n) * FREQ * DT
    T = t[-1] + FREQ * DT
    w = 2 * np.pi / T
    c = START + np.array([-r, 0.0, -1.5])
    tab = np.zeros((n, 11))
    tab[:, 0], tab[:, 1], tab[:, 2] = c[0] + r * np.cos(w * t), c[1] + r * np.sin(w * t), c[2] - 0.1 * t
    tab[:, 3], tab[:, 4], tab[:, 5] = -r * w * np.sin(w * t), r * w * np.cos(w * t), -0.1
    tab[:, 6], tab[:, 7] = -r * w * w * np.cos(w * t), -r * w * w * np.sin(w * t)
    tab[:, 9] = 2 * np.pi * turns_yaw * t / T
    tab[:, 10] = 7
    return tab


def hover_table():
    return np.array([[START[0] + 0.2, START[1] - 0.1, -1.0, 0, 0, 0, 0, 0, 0, 0.4, 0]])


def figure_eight_table(n=900, a=1.5):
    """Lissajous figure-eight with zero acceleration columns."""
    t = np.arange(n) * FREQ * DT
    w = 2 * np.pi / (n * FREQ * DT)
    tab = np.zeros((n, 11))
    tab[:, 0], tab[:, 1], tab[:, 2] = START[0] + a * np.sin(w * t), START[1] + a * np.sin(2 * w * t) / 2, -1.2
    tab[:, 3], tab[:, 4] = a * w * np.cos(w * t), a * w * np.cos(2 * w * t)
    tab[:, 9] = np.arctan2(tab[:, 4], tab[:, 3])
    return tab


def random_walk_table(n=500, seed=5):
    """Set-points that are not dynamically consistent: a random walk of positions with unrelated v / a / yaw columns."""
    rng = np.random.default_rng(seed)
    tab = np.zeros((n, 11))
    tab[:, :3] = START + np.array([0, 0, -1.0]) + np.cumsum(rng.normal(0, 0.02, (n, 3)), axis=0)
    tab[:, 3:6] = rng.normal(0, 0.3, (n, 3))
    tab[:, 6:9] = rng.normal(0, 0.5, (n, 3))
    tab[:, 9] = np.cumsum(rng.normal(0, 0.05, n))
    tab[:, 10] = rng.integers(0, 5, n)
    return tab


def lissajous_table(n, rng):
    """Smooth random table that starts at rest on the start point: a climb to 0.5-1.5 m with a horizontal Lissajous drift."""
    t = np.arange(n) * FREQ * DT
    amp, w = rng.uniform(0.3, 2.0, 3), rng.uniform(0.2, 0.8, 3)
    amp[2] = rng.uniform(0.25, 0.75)
    sign = np.array([rng.choice([-1.0, 1.0]), rng.choice([-1.0, 1.0]), -1.0])
    tab = np.zeros((n, 11))
    for k in range(3):                                   # p = start + s amp (1 - cos w t): zero velocity at t = 0
        tab[:, k] = START[k] + sign[k] * amp[k] * (1 - np.cos(w[k] * t))
        tab[:, 3 + k] = sign[k] * amp[k] * w[k] * np.sin(w[k] * t)
        tab[:, 6 + k] = sign[k] * amp[k] * w[k] ** 2 * np.cos(w[k] * t)
    tab[:, 9] = rng.uniform(-1, 1) + 0.3 * t
    return tab


def _vehicle(vals=None, b=None):
    from oracle import flight_np
    if vals is None:
        return flight_np.Vehicle()
    kw = {k: getattr(flight_np.Vehicle(), k) for k in flight_np.Vehicle.__dataclass_fields__}
    for k, name in enumerate(flight_np.Vehicle.GAIN_NAMES):
        kw[name] = vals[k, b]
    kw["mass"], kw["inertia"] = vals[11, b], vals[12:15, b]
    return flight_np.Vehicle(**kw)


def _gap(log_xyz, boxes):
    """Smallest distance of the oracle path to any box face (signed Chebyshev distance, absolute)."""
    gap = np.inf
    for q in np.asarray(boxes, float).reshape(-1, 6):
        P = log_xyz
        d = np.maximum.reduce([q[0] - P[:, 0], P[:, 0] - q[1], q[2] - P[:, 1], P[:, 1] - q[3], q[4] - P[:, 2], P[:, 2] - q[5]])
        gap = min(gap, np.abs(d).min())
    return gap


def _compare(met, X, ref, what, flags=True, boxes=None):
    """One rollout (metrics [8], final state [13]) against a C-oracle result."""
    dp = np.abs(X[:3] - ref["X"][:3]).max()
    da = rotation_angle(X[3:7], ref["X"][3:7])
    assert dp < POS_TOL and da < ANG_TOL, f"{what}: |dpos| {dp:.2e} m, attitude {da:.2e} rad"
    assert met[7] == ref["periods"], what
    for k, name in ((2, "rmse"), (3, "mean_err"), (4, "max_err")):
        assert abs(met[k] - ref[name]) < POS_TOL, f"{what}: {name} {met[k]} vs {ref[name]}"
    if "final_dist" in ref:
        assert abs(met[0] - ref["final_dist"]) < POS_TOL, what
    assert met[5] == 0, what
    if flags and (boxes is None or ref["log"] is None or _gap(ref["log"][:, :3], boxes) >= POS_TOL):
        assert met[1] == float(ref["collision"]) and met[6] == ref["first_collision_tick"], what
        return True
    return False


def _fly(dev, plan, B, n_ticks, start=START, goal=GOAL, **kw):
    import torch
    from uav_ac_b200 import kernels
    s = torch.as_tensor(np.asarray(start, float), dtype=torch.float64).to(dev).contiguous()
    g = None if goal is None else torch.as_tensor(np.asarray(goal, float), dtype=torch.float64).to(dev).contiguous()
    res = kernels.rollout(plan, B, n_ticks, start=s, goal=g, **kw)
    torch.cuda.synchronize()
    return res


# ------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def nat():
    from uav_ac_b200 import _native
    if not os.path.exists(_native.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _native


def test_table_set_layout_matches_the_header(nat, tmp_path):
    probe = tmp_path / "probe.c"
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "uavb.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %d\\n",'
                     'sizeof(uavb_table_set), offsetof(uavb_table_set, rows), offsetof(uavb_table_set, offsets), offsetof(uavb_table_set, table_index),'
                     'offsetof(uavb_table_set, n_tables), offsetof(uavb_table_set, shared_rows), UAVB_TARGET_ROW_BYTES);return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    T = nat.TableSet
    assert got == [ctypes.sizeof(T), T.rows.offset, T.offsets.offset, T.table_index.offset, T.n_tables.offset, T.shared_rows.offset,
                   nat.TARGET_ROW_BYTES]


def test_table_entry_points_validate_their_arguments(nat):
    import torch
    L = nat.lib()
    null = ctypes.c_void_p(None)
    one = ctypes.c_void_p(8)                                     # non-NULL dummy; validation happens before any dereference

    def args():
        a = nat.RolloutArgs()
        a.B, a.n_ticks, a.inner_per_outer = 4, 100, 10
        a.veh = nat.default_vehicle()
        a.start = one
        return a

    def tset(**kw):
        t = nat.TableSet()
        t.rows, t.offsets, t.n_tables = one, one, 4
        for k, v in kw.items():
            setattr(t, k, v)
        return t

    def call(a, t):
        return L.uavb_rollout_tables_f32(ctypes.byref(a), ctypes.byref(t) if t is not None else None, null)

    assert call(args(), tset(rows=null)) == -1 and b"rows" in L.uavb_last_error()                     # NULL rows
    assert call(args(), None) == -1
    assert call(args(), tset(n_tables=0)) == -1 and b"n_tables" in L.uavb_last_error()               # n_tables < 1
    assert call(args(), tset(n_tables=3)) == -1                                                       # no index: n_tables == B
    for field, value in (("seg_coeffs", one), ("seg_rows", one), ("seg_table", one), ("seg_yaw0", one), ("mission_seg_begin", one),
                         ("mission_seg_count", one), ("shared_targets", one), ("n_seg_shared", 1), ("n_target_rows", 5)):
        a = args()
        setattr(a, field, value)
        assert call(a, tset()) == -1 and b"mission-segment" in L.uavb_last_error(), field              # a set segment field
    assert call(args(), tset(offsets=null, shared_rows=5, table_index=one)) == -1 and b"shared" in L.uavb_last_error()
    assert call(args(), tset(shared_rows=5)) == -1                                                    # shared table with offsets
    assert call(args(), tset(shared_rows=-1)) == -1
    a = args()
    a.inner_per_outer = 0
    assert call(a, tset()) == -1 and b"inner_per_outer" in L.uavb_last_error()
    assert L.uavb_table_targets_f64(null, 4, one, null) == -1 and L.uavb_table_targets_f64(one, -1, one, null) == -1
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible: the ENODEVICE leg only applies to GPU-less hosts")
    assert call(args(), tset()) == -3 and call(args(), tset(offsets=null, n_tables=0, shared_rows=7)) == -3       # UAVB_ENODEVICE
    assert L.uavb_table_targets_f64(one, 4, one, null) == -3


def test_plan_tables_rejects_bad_shapes_and_indices():
    import torch
    from uav_ac_b200 import kernels
    good = np.zeros((5, 11))
    with pytest.raises(ValueError):
        kernels.plan_tables(np.zeros((5, 10)))                                 # 10 columns
    with pytest.raises(ValueError):
        kernels.plan_tables(np.zeros((0, 11)))                                 # no rows
    with pytest.raises(ValueError):
        kernels.plan_tables([good, np.zeros((0, 11))])
    with pytest.raises(ValueError):
        kernels.plan_tables(np.zeros((2, 3, 4, 11)))
    with pytest.raises(ValueError):
        kernels.plan_tables([good, np.zeros(11)])
    with pytest.raises(ValueError):
        kernels.plan_tables([])
    with pytest.raises(ValueError):
        kernels.plan_tables([good, good], table_index=[0, 2])                  # index out of range
    with pytest.raises(ValueError):
        kernels.plan_tables([good, good], table_index=[-1, 0])
    with pytest.raises(ValueError):
        kernels.plan_tables([good, good], table_index=np.zeros((2, 2), dtype=int))
    with pytest.raises(ValueError):
        kernels.plan_tables([good, good], table_index=torch.zeros(2))          # not integer


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_reference_table_through_fly_trajectory_matches_reference_closed_loop(cuda, golden):
    """planning["v3_table"] is the reference's own table; closed_loop_v3 its own objects' closed loop on it."""
    from uav_ac_b200.simulation.batched_sim import BatchedSimulation
    tab, gold = golden["planning"]["v3_table"], golden["closed_loop_v3"]
    sim = BatchedSimulation(batch=1, device=cuda)
    res = sim.fly_trajectory(tab, 10, log_stride=10)
    assert res.n_ticks == 10 * len(tab) == 10760
    X = res.log[:, :, 0].double().cpu().numpy()
    assert X.shape == gold["X"].shape
    dp, da = np.abs(X[:, :3] - gold["X"][:, :3]).max(), rotation_angle(X[:, 3:7], gold["X"][:, 3:7]).max()
    print(f"per-period states: max |dpos| {dp:.2e} m, attitude {da:.2e} rad")
    assert dp < POS_TOL and da < ANG_TOL
    m = res.metrics[0].double().cpu().numpy()
    for k, name in ((0, "final_dist"), (2, "rmse"), (3, "mean_err"), (4, "max_err")):
        assert abs(m[k] - float(gold[name])) < POS_TOL, name
    assert m[1] == float(gold["collision"]) and m[6] == float(gold["first_collision_tick"]) and m[7] == len(tab) and m[5] == 0
    fine = sim.fly_trajectory(tab, 10, n_ticks=2000, log_stride=1).log[:, :, 0].double().cpu().numpy()
    ref = gold["fine"][:, :13]
    assert np.abs(fine[:, :3] - ref[:, :3]).max() < POS_TOL and rotation_angle(fine[:, 3:7], ref[:, 3:7]).max() < ANG_TOL


@pytest.mark.gpu
def test_tables_that_are_not_min_snap_output_match_the_c_oracle(cuda):
    """Circle with yaw through three turns, one-row hover, figure-eight with zero accelerations, a random walk; flown as a shared
    table and as per-rollout tables in one batch; tick counts below, at and beyond frequency x N (index clamp)."""
    from oracle import c_port
    from uav_ac_b200 import kernels
    tables = {"circle": circle_table(2000), "hover": hover_table(), "eight": figure_eight_table(), "walk": random_walk_table()}
    boxes = np.array([[0.5, 1.5, 8.5, 9.5, -2.5, -1.0],                     # on the circle: a hit with an exact first tick
                      [5.0, 6.0, 0.0, 1.0, -3.0, -1.0]])                    # away from every path
    import torch
    obs = torch.tensor(boxes, dtype=torch.float32, device=cuda)
    exact = 0
    for name, tab in tables.items():
        N = len(tab)
        for n_ticks in (FREQ * N - 37 if N > 4 else 3, FREQ * N, FREQ * N + 503):
            ref = c_port.closed_loop(_vehicle(), tab, START, freq=FREQ, n_ticks=n_ticks, obstacles=boxes, goal=GOAL, log_stride=1)
            res = _fly(cuda, kernels.plan_tables(tab), 2, n_ticks, obstacles=obs)
            met, X = res.metrics.double().cpu().numpy(), res.state.double().cpu().numpy()
            exact += _compare(met[0], X[:, 0], ref, f"{name} shared n={n_ticks}", boxes=boxes)
            assert np.array_equal(met[0], met[1])
    assert exact >= 6
    # the four tables at once, one per rollout (per-rollout kernel), past the end of the longest
    plan = kernels.plan_tables(list(tables.values()))
    n_ticks = FREQ * plan.max_rows + 200
    res = _fly(cuda, plan, 4, n_ticks, obstacles=obs)
    met, X = res.metrics.double().cpu().numpy(), res.state.double().cpu().numpy()
    for b, (name, tab) in enumerate(tables.items()):
        ref = c_port.closed_loop(_vehicle(), tab, START, freq=FREQ, n_ticks=n_ticks, obstacles=boxes, goal=GOAL, log_stride=1)
        _compare(met[b], X[:, b], ref, f"{name} per-rollout", boxes=boxes)
    print(f"collision flags exact in {exact} shared flights")


def _per_rollout_setup(dev, B=10_001, T=64, seed=17):
    import torch
    from uav_ac_b200 import kernels, _native as nat
    rng = np.random.default_rng(seed)
    lengths = np.concatenate(([1, 2000], rng.integers(1, 2001, T - 2)))
    tables = [lissajous_table(int(n), rng) for n in lengths]
    index = rng.integers(0, T, B)
    index[0], index[-1] = 0, 1
    sc = kernels.mc_uniform(31, B, [0.8] * 11 + [0.9] * 4, [1.2] * 11 + [1.1] * 4, device=dev)
    v = nat.default_vehicle()
    base = torch.tensor(list(v.gains) + [v.mass] + list(v.inertia), dtype=torch.float32, device=dev)[:, None]
    vals = (sc * base).contiguous()
    wind = kernels.mc_uniform(32, B, [-0.08] * 3, [0.08] * 3, device=dev)
    ctr = rng.uniform([1.0, 4.0, -3.5], [5.0, 10.0, -0.5], (8, 4, 3))
    half = rng.uniform(0.2, 0.8, (8, 4, 3))
    boxes = np.stack((ctr[..., 0] - half[..., 0], ctr[..., 0] + half[..., 0], ctr[..., 1] - half[..., 1], ctr[..., 1] + half[..., 1],
                      ctr[..., 2] - half[..., 2], ctr[..., 2] + half[..., 2]), axis=-1).astype(np.float32)
    sets = rng.integers(0, 8, B)
    kw = dict(mc_gains=vals[:11].contiguous(), mc_mass=vals[11].contiguous(), mc_inertia=vals[12:15].contiguous(), mc_wind=wind,
              obstacles=torch.tensor(boxes, device=dev), obstacle_set=torch.tensor(sets, dtype=torch.int32, device=dev))
    return tables, index, vals, wind, boxes, sets, kw


@pytest.mark.gpu
def test_per_rollout_tables_match_the_c_oracle_on_a_sample(cuda):
    """64 tables of 1 to 2 000 rows, B = 10 001 (the last pair re-flies its first lane), random table_index, mass / inertia / gains /
    wind overrides and per-rollout obstacle sets; >= 64 sampled rollouts against the C oracle on their own table and vehicle."""
    from oracle import c_port
    from uav_ac_b200 import kernels
    tables, index, vals, wind, boxes, sets, kw = _per_rollout_setup(cuda)
    B = len(index)
    plan = kernels.plan_tables(tables, table_index=index, device=cuda)
    assert plan.rows_per_table[0] == 1 and plan.max_rows == 2000
    n_ticks = FREQ * plan.max_rows
    goal = plan.goals(B)
    res = _fly(cuda, plan, B, n_ticks, goal=goal.cpu().numpy(), **kw)
    met, X = res.metrics.double().cpu().numpy(), res.state.double().cpu().numpy()
    assert np.isfinite(met).all() and (met[:, 5] == 0).all()
    assert 0.02 < met[:, 1].mean() < 0.98                                          # both outcomes are exercised
    vals_h, wind_h = vals.double().cpu().numpy(), wind.double().cpu().numpy()
    sample = sorted(set([0, 1, B - 2, B - 1] + list(np.random.default_rng(3).choice(B, 64, replace=False))))
    exact = 0
    for b in sample:
        tab = tables[index[b]]
        ref = c_port.closed_loop(_vehicle(vals_h, b), tab, START, freq=FREQ, n_ticks=n_ticks, obstacles=boxes[sets[b]].astype(float),
                                 goal=tab[-1, :3], wind=wind_h[:, b], log_stride=1)
        exact += _compare(met[b], X[:, b], ref, f"rollout {b} (table {index[b]}, {len(tab)} rows)", boxes=boxes[sets[b]])
    print(f"{len(sample)} sampled rollouts within budget; collision flags exact in {exact}")
    assert exact >= len(sample) // 2


@pytest.mark.gpu
def test_per_rollout_tables_are_invariant_bit_for_bit(cuda):
    """Alone, at another B or with another partner; n_slices 1 / 3 / 17; three chunked launches; tensor vs per-thread log stores."""
    import torch
    from uav_ac_b200 import kernels
    tables, index, vals, wind, boxes, sets, kw = _per_rollout_setup(cuda, B=1001, T=16, seed=23)
    B = len(index)
    plan = kernels.plan_tables(tables, table_index=index, device=cuda)
    n = 3007                                                                   # not a multiple of the outer period
    whole = _fly(cuda, plan, B, n, **kw)

    def sub(ids):
        ids_t = torch.tensor(ids, dtype=torch.long, device=cuda)
        p = kernels.plan_tables(tables, table_index=index[ids], device=cuda)
        k = dict(mc_gains=kw["mc_gains"][:, ids_t].contiguous(), mc_mass=kw["mc_mass"][ids_t].contiguous(),
                 mc_inertia=kw["mc_inertia"][:, ids_t].contiguous(), mc_wind=kw["mc_wind"][:, ids_t].contiguous(), obstacles=kw["obstacles"],
                 obstacle_set=kw["obstacle_set"][ids_t].contiguous())
        return _fly(cuda, p, len(ids), n, **k)

    for ids in ([5], [7, 5], [5, 7, 900], list(range(1000, 0, -3))):
        r = sub(ids)
        for j, b in enumerate(ids):
            assert torch.equal(r.state[:, j], whole.state[:, b]) and torch.equal(r.metrics[j], whole.metrics[b]), (ids, b)
    for s in (1, 3, 17):
        r = _fly(cuda, plan, B, n, n_slices=s, **kw)
        assert torch.equal(r.state, whole.state) and torch.equal(r.metrics, whole.metrics), s
    a = _fly(cuda, plan, B, 1003, want_carry=True, **kw)
    b = _fly(cuda, plan, B, 1000, carry=a.carry, resume=True, want_carry=True, **kw)
    c = _fly(cuda, plan, B, n - 2003, carry=b.carry, resume=True, **kw)
    assert torch.equal(c.state, whole.state) and torch.equal(c.metrics, whole.metrics)
    idx4 = index[:1000]
    p4 = kernels.plan_tables(tables, table_index=idx4, device=cuda)
    k4 = {k: (v[..., :1000].contiguous() if k.startswith("mc_") or k == "obstacle_set" else v) for k, v in kw.items()}
    tma = _fly(cuda, p4, 1000, 1500, log_stride=7, log_tma=0, **k4)
    thr = _fly(cuda, p4, 1000, 1500, log_stride=7, log_tma=-1, **k4)
    assert torch.equal(tma.log, thr.log) and torch.equal(tma.state, thr.state)


@pytest.mark.gpu
def test_shared_table_against_replicated_and_mission_plan_against_its_sampled_table(cuda):
    import torch
    from helpers import lab_course_plan
    from uav_ac_b200 import kernels
    from uav_ac_b200.simulation.scene import LAB_COURSE_OBSTACLES
    obs = torch.tensor(LAB_COURSE_OBSTACLES, dtype=torch.float32, device=cuda)
    tab = circle_table()
    B, n = 64, FREQ * len(tab)
    shared = _fly(cuda, kernels.plan_tables(tab), B, n, obstacles=obs)
    repl = _fly(cuda, kernels.plan_tables(tab, table_index=np.zeros(B, dtype=np.int32)), B, n, obstacles=obs)
    dp = float((shared.state[:3].double() - repl.state[:3].double()).abs().max())
    print(f"shared vs replicated table: max |dpos| {dp:.2e} m")
    assert dp < 1e-6 and torch.equal(shared.metrics[:, 1], repl.metrics[:, 1])
    # the lab_course mission as a MissionPlan and as its K3-sampled table (the reference's get_trajectory() stitching, main.py:80-84)
    plan = lab_course_plan(cuda, 3.0)
    n_take = int(plan.seg_rows[:1].sum())
    n_rows = int(plan.total_rows.sum())
    seg_off = torch.tensor([0, 1, plan.seg_rows.numel()], dtype=torch.int32, device=cuda)
    row_off = torch.tensor([0, n_take, n_rows], dtype=torch.int32, device=cuda)
    k3 = kernels.minsnap_sample(plan.seg_coeffs, plan.times, seg_off, plan.seg_rows, row_off, plan.dt)
    a = _fly(cuda, plan, 4, 10 * n_rows, obstacles=obs)
    b = _fly(cuda, kernels.plan_tables(k3), 4, 10 * n_rows, obstacles=obs)
    d = (a.metrics.double() - b.metrics.double()).abs().max(dim=0).values.cpu().numpy()
    print(f"MissionPlan vs its K3 table: metric differences {d}")
    assert d.max() < 1e-5


@pytest.mark.gpu
def test_table_options_flown_path_floor_empty_launches_and_nan(cuda, golden):
    import torch
    from oracle import c_port, flight_np
    from uav_ac_b200 import kernels, _native as nat
    from uav_ac_b200.simulation.batched_sim import BatchedSimulation
    # flown-path list of the viewer (mujoco_sim.py:201-218) against the NumPy oracle: same samples, same positions
    tab = golden["planning"]["v3_table"]
    sim = BatchedSimulation(batch=2, device=cuda)
    res = sim.fly_trajectory(tab, 10, record_actual_trajectory=True)
    gate = float(sim.mission_waypoints[1][2])
    ref = flight_np.closed_loop(flight_np.Vehicle(), tab, START, goal=GOAL, traj_gate_z=gate, obstacles=sim.obstacles)
    cnt = int(res.traj_count[0])
    assert cnt == len(ref["traj_ticks"]) == int(res.traj_count[1])
    P = res.traj[:cnt, :, 0].double().cpu().numpy()
    assert np.abs(P - ref["traj"]).max() < POS_TOL
    # per-rollout tables with the flown-path list: both drones' own tables
    two = sim.fly_trajectory([tab, tab[:400]], 10, table_index=[1, 0], record_actual_trajectory=True)
    assert int(two.traj_count[1]) == cnt and torch.equal(two.traj[:cnt, :, 1], res.traj[:cnt, :, 0])
    # the floor (ground_z): a hover table starting on the ground
    hov = hover_table()
    refg = c_port.closed_loop(_vehicle(), hov, START, freq=FREQ, n_ticks=1500, goal=GOAL, ground_z=START[2])
    rg = _fly(cuda, kernels.plan_tables(hov), 2, 1500, ground_z=float(START[2]))
    _compare(rg.metrics[0].double().cpu().numpy(), rg.state[:, 0].double().cpu().numpy(), refg, "hover with floor", flags=False)
    # n_ticks = 0 and B = 0
    plan = kernels.plan_tables([hov, circle_table()], table_index=[1, 0, 1])
    r0 = _fly(cuda, plan, 3, 0)
    assert (r0.metrics[:, 7] == 0).all() and torch.allclose(r0.state[:3].double().T, torch.tensor(START, device=cuda).expand(3, 3))
    empty = kernels.plan_tables([hov], table_index=np.zeros(0, dtype=np.int32))
    rb = _fly(cuda, empty, 0, 100)
    assert rb.metrics.shape == (0, nat.N_METRICS)
    # a NaN row: UAVB_ROLLOUT_NONFINITE, the other rollout unaffected
    bad = circle_table(200)
    bad[50, 0] = np.nan
    rn = _fly(cuda, kernels.plan_tables([bad, circle_table(200)]), 2, 2000)
    m = rn.metrics.cpu().numpy()
    assert int(m[0, 5]) & 1 and m[1, 5] == 0
    # fp64 has no table form
    with pytest.raises(ValueError):
        _fly(cuda, kernels.plan_tables(hov), 1, 10, dtype=torch.float64)
