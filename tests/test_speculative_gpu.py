"""Speculative stretches of the metrics-only pair kernels (rollout_pair.cuh): a non-watching stretch flies the branch-free tick from a
shared-memory checkpoint and replays with the exact body when some lane of the warp would have taken the rotor-limit or the
large-rotation path.  Results must be the exact body's bit for bit, whatever the rollback rate.

The exact body is forced in the same process through the development entry point uavb_dev_speculation (not part of uavb.h).
Workloads: a hover (no rare path), the bench workload (shared lab_course table, Monte-Carlo vehicles, boxes), wind plus +-50 % gains
(rollback-heavy), and a tumbling low-inertia vehicle that takes the large-rotation path; the last two fly per-rollout tables too."""
import ctypes

import numpy as np
import pytest

from helpers import hover_table, lab_course_plan, mc_arrays, rough_mc

START = np.array([1.0, 7.0, -0.021])            # lab_course start
FREQ = 10
SMALL_ROT_W = 44.72                              # |w| above which the exact tick takes the large-rotation map (veh_setup.cuh, dt = 1 ms)


@pytest.fixture(scope="module")
def spec(cuda):
    """force(flag): fly every stretch of the speculative kernels with the exact body (1) or speculate (0)."""
    from uav_ac_b200 import _native as nat
    fn = nat.lib().uavb_dev_speculation
    fn.argtypes = [ctypes.c_int]
    fn.restype = ctypes.c_int

    def force(flag):
        assert fn(int(flag)) == 0
    yield force
    force(0)


def _bits(t):
    import torch
    return t.contiguous().view(torch.int32)


def _same(a, b):
    """Bit-identical metrics and (when present) final state: NaN patterns included."""
    import torch
    ok = torch.equal(_bits(a.metrics), _bits(b.metrics))
    if a.state is not None:
        ok = ok and torch.equal(_bits(a.state), _bits(b.state))
    return ok


def _fly(plan, B, n_ticks, dev, **kw):
    import torch
    from uav_ac_b200 import kernels
    kw.setdefault("start", torch.tensor(START, dtype=torch.float64, device=dev))
    res = kernels.rollout(plan, B, n_ticks, **kw)
    torch.cuda.synchronize()
    return res


def _both(spec, plan, B, n_ticks, dev, **kw):
    spec(1)
    try:
        exact = _fly(plan, B, n_ticks, dev, **kw)
    finally:
        spec(0)
    fast = _fly(plan, B, n_ticks, dev, **kw)
    return fast, exact


def _hover_table():
    return hover_table(START)


def _bench_setup(dev, B):
    import torch
    import bench_workloads as wl
    from uav_ac_b200 import _native as nat
    from uav_ac_b200 import kernels
    plan, kw = wl.lab_course(kernels, dev)
    mc = wl.mc_vehicle_arrays(kernels, nat, dev, B)
    kw = dict(kw, mc_gains=mc[:11], mc_mass=mc[11], mc_inertia=mc[12:15], want_state=True)
    return plan, 10 * int(plan.total_rows.sum()), kw, torch


_rough = rough_mc


@pytest.mark.gpu
def test_hover_is_bit_identical(cuda, spec):
    from uav_ac_b200 import kernels
    plan = kernels.plan_tables(_hover_table(), device=cuda)
    fast, exact = _both(spec, plan, 4099, 3000, cuda)
    assert np.isfinite(fast.metrics.cpu().numpy()).all()
    assert _same(fast, exact)


@pytest.mark.gpu
def test_bench_workload_is_bit_identical(cuda, spec):
    plan, n_ticks, kw, torch = _bench_setup(cuda, 20_000)
    fast, exact = _both(spec, plan, 20_000, n_ticks, cuda, **kw)
    assert (fast.metrics[:, 5] == 0).all()
    assert _same(fast, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("tumble", [False, True])
def test_rollback_heavy_workloads_are_bit_identical_shared_and_per_rollout(cuda, spec, tumble):
    import torch
    from uav_ac_b200 import kernels
    B = 6001
    kw = _rough(cuda, B, tumble=tumble)
    tab = _hover_table()
    tab[0, 9] = 3.0 if tumble else 0.4
    shared = kernels.plan_tables(tab, device=cuda)
    fast, exact = _both(spec, shared, B, 3000, cuda, **kw)
    assert _same(fast, exact)
    # per-rollout tables: the same table shifted by up to +-0.3 m per copy, 64 copies
    rng = np.random.default_rng(4)
    tabs = np.repeat(tab[None], 64, axis=0)
    tabs[:, 0, :3] += rng.uniform(-0.3, 0.3, (64, 3))
    idx = torch.tensor(rng.integers(0, 64, B), dtype=torch.int32, device=cuda)
    per = kernels.plan_tables(tabs, table_index=idx, device=cuda)
    fast, exact = _both(spec, per, B, 3000, cuda, **kw)
    assert _same(fast, exact)
    if tumble:
        # the large-rotation path is taken: the state log (an exact-body kernel flying the same vehicles) shows |w| above the bound
        log = _fly(shared, 64, 3000, cuda, log_stride=1, **{k: v[..., :64].contiguous() for k, v in kw.items()}).log
        w = log.reshape(3000, 13, 64)[:, 10:13].double().norm(dim=1)
        assert int((w[:, ::2] > SMALL_ROT_W).sum()) > 1000


@pytest.mark.gpu
def test_rollback_heavy_batch_is_invariant_across_position_slicing_and_resume(cuda, spec):
    import torch
    from uav_ac_b200 import kernels
    B = 3001
    kw = _rough(cuda, B, seed=5, tumble=True)
    plan = kernels.plan_tables(_hover_table(), device=cuda)
    n = 3007                                                                   # not a multiple of the outer period
    whole = _fly(plan, B, n, cuda, **kw)

    def sub(ids):
        ids_t = torch.tensor(ids, dtype=torch.long, device=cuda)
        return _fly(plan, len(ids), n, cuda, **{k: v[..., ids_t].contiguous() for k, v in kw.items()})

    for ids in ([6], [7, 6], [6, 7, 2900], list(range(3000, 0, -7))):
        r = sub(ids)
        for j, b in enumerate(ids):
            assert torch.equal(_bits(r.state[:, j]), _bits(whole.state[:, b])) and torch.equal(_bits(r.metrics[j]), _bits(whole.metrics[b])), (ids, b)
    for s in (1, 3, 17):
        assert _same(_fly(plan, B, n, cuda, n_slices=s, **kw), whole), s
    a = _fly(plan, B, 1003, cuda, want_carry=True, **kw)
    b = _fly(plan, B, 1000, cuda, carry=a.carry, resume=True, want_carry=True, **kw)
    c = _fly(plan, B, n - 2003, cuda, carry=b.carry, resume=True, **kw)
    assert _same(c, whole)


@pytest.mark.gpu
def test_speculative_kernels_match_the_c_oracle_on_a_sample(cuda, spec):
    """Shared lab_course table and per-rollout copies of it, wind and +-50 % gains: sampled rollouts against the fp64 C oracle."""
    import torch
    from oracle import c_port, flight_np
    from uav_ac_b200 import kernels
    plan = lab_course_plan(cuda, 3.0)
    n_rows = int(plan.total_rows.sum())
    seg_off = torch.tensor([0, 1, plan.seg_rows.numel()], dtype=torch.int32, device=cuda)
    n_take = int(plan.seg_rows[:1].sum())
    row_off = torch.tensor([0, n_take, n_rows], dtype=torch.int32, device=cuda)
    table = kernels.minsnap_sample(plan.seg_coeffs, plan.times, seg_off, plan.seg_rows, row_off, plan.dt).cpu().numpy()
    B, n_ticks = 2048, FREQ * n_rows
    rng = np.random.default_rng(9)
    gains, wind = rng.uniform(0.5, 1.5, (B, 11)), rng.uniform(-0.08, 0.08, (B, 3))
    kw = mc_arrays(cuda, B, gain_scale=gains, wind=wind)
    goal = torch.tensor(table[-1, :3], dtype=torch.float64, device=cuda)
    for p in (kernels.plan_tables(table, device=cuda), kernels.plan_tables(np.repeat(table[None], 2, axis=0),
                                                                          table_index=torch.arange(B, device=cuda, dtype=torch.int32) % 2, device=cuda)):
        res = _fly(p, B, n_ticks, cuda, goal=goal, **kw)
        met, X = res.metrics.double().cpu().numpy(), res.state.double().cpu().numpy()
        for b in (0, 1, 777, B - 1):
            v = flight_np.Vehicle()
            f = {k: getattr(v, k) for k in flight_np.Vehicle.__dataclass_fields__}
            for k, name in enumerate(flight_np.Vehicle.GAIN_NAMES):
                f[name] = float(np.float32(getattr(v, name) * gains[b, k]))
            ref = c_port.closed_loop(flight_np.Vehicle(**f), table, START, freq=FREQ, n_ticks=n_ticks, goal=table[-1, :3],
                                     wind=np.float32(wind[b]).astype(float))
            assert np.abs(X[:3, b] - ref["X"][:3]).max() < 1e-4, b
            assert met[b, 7] == ref["periods"] and met[b, 5] == 0, b
            for k, name in ((2, "rmse"), (3, "mean_err"), (4, "max_err"), (0, "final_dist")):
                assert abs(met[b, k] - ref[name]) < 1e-4, (b, name)
