"""K2 flying caller-supplied trajectory tables: CUDA-event timing of four arms at 1e5 rollouts with the Monte-Carlo set-up of
bench.py (perturbed gains / mass / inertia from the counter-based generator, the 4 lab_course AABBs, metrics only), one JSON line
per arm, with the card's name and power limit read in the same run.

    python tools/table_probe.py [--rollouts 100000] [--reps 5] [--arms a,b,c,d] [--lib PATH] [--out FILE]

  a  the lab_course K3 table at v = 3 (1 076 rows) as ONE shared caller table (the shared-table kernel of the headline workload)
  b  64 distinct tables (the same table shifted vertically by up to +-0.3 m) mapped by table_index
  c  one table per rollout (1e5 x 1 076 rows x 56 B = 6.0 GB of set-point records, larger than L2)
  d  the same batch as per-rollout MissionPlan missions (the reference arm: splines evaluated in fp64 on the fly)

A 256 MB buffer is written between timed passes (L2 flush).  steps/s = rollouts x ticks / kernel time; table_bytes_per_s = the
set-point records the kernel reads (56 B per rollout and outer period) / kernel time -- for arm a every rollout reads the same
60 kB, so that figure is L1/L2 traffic, not HBM.  --lib flies another build of the library, e.g. a parent commit's libuavb.so.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                               text=True, timeout=20).stdout.strip()
        limit = float(limit.splitlines()[0])
    except Exception:                                  # noqa: BLE001 -- reported as unknown, never guessed
        limit = None
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rollouts", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--arms", default="a,b,c,d")
    ap.add_argument("--lib", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from uav_ac_b200 import _native as nat
    if args.lib:
        nat.LIB_PATH = os.path.abspath(args.lib)
    from uav_ac_b200 import kernels
    from uav_ac_b200.simulation.scene import LAB_COURSE_GOAL, LAB_COURSE_OBSTACLES, LAB_COURSE_START, LAB_COURSE_WAYPOINTS
    if not torch.cuda.is_available():
        raise SystemExit("table_probe: no CUDA device (a timing needs the GPU)")
    dev = torch.device("cuda", 0)
    name, limit = card()
    B = args.rollouts
    f64 = dict(dtype=torch.float64, device=dev)
    W = torch.tensor(LAB_COURSE_WAYPOINTS, **f64)
    v3 = torch.tensor([3.0], **f64)
    shared_plan = kernels.plan_missions([(W[None, :2].contiguous(), v3), (W[None, 1:].contiguous(), v3)], 0.01, shared=True)
    n_take, n_rows = int(shared_plan.seg_rows[:1].sum()), int(shared_plan.total_rows.sum())
    seg_off = torch.tensor([0, 1, shared_plan.seg_rows.numel()], dtype=torch.int32, device=dev)
    row_off = torch.tensor([0, n_take, n_rows], dtype=torch.int32, device=dev)
    k3 = kernels.minsnap_sample(shared_plan.seg_coeffs, shared_plan.times, seg_off, shared_plan.seg_rows, row_off, shared_plan.dt)
    n_ticks = 10 * n_rows
    veh = nat.default_vehicle()
    base = torch.tensor(list(veh.gains) + [veh.mass] + list(veh.inertia), dtype=torch.float32, device=dev)[:, None]
    mc = (kernels.mc_uniform(1, B, [0.8] * 11 + [0.9] * 4, [1.2] * 11 + [1.1] * 4) * base).contiguous()
    kw = dict(start=torch.tensor(LAB_COURSE_START, **f64), goal=torch.tensor(LAB_COURSE_GOAL, **f64),
              obstacles=torch.tensor(LAB_COURSE_OBSTACLES, dtype=torch.float32, device=dev), want_state=False,
              mc_gains=mc[:11], mc_mass=mc[11], mc_inertia=mc[12:15])
    gen = torch.Generator(device=dev).manual_seed(7)

    def shifted(T):
        """T copies of the K3 table, copy t shifted vertically by a constant of up to +-0.3 m: [T, n_rows, 11] f64 (a horizontal
        offset of the take-off rows tips a drone that still sits on the start height -- the fp64 oracle diverges as well)."""
        shift = (torch.rand((T, 1), generator=gen, device=dev, dtype=torch.float64) - 0.5) * 0.6
        out = k3[None].repeat(T, 1, 1)
        out[:, :, 2] += shift
        return out

    def plan_for(arm):
        if arm == "a":
            return kernels.plan_tables(k3), n_rows * 56
        if arm == "b":
            idx = torch.randint(0, 64, (B,), generator=gen, device=dev, dtype=torch.int32)
            return kernels.plan_tables(shifted(64), table_index=idx), 64 * n_rows * 56
        if arm == "c":
            return kernels.plan_tables(shifted(B)), B * n_rows * 56
        wp = W[None].repeat(B, 1, 1)
        wp[:, 1:, :3] += (torch.rand((B, 1, 3), generator=gen, device=dev, dtype=torch.float64) - 0.5) * 1e-3
        vel = torch.full((B,), 3.0, **f64)
        return kernels.plan_missions([(wp[:, :2].contiguous(), vel), (wp[:, 1:].contiguous(), vel)], 0.01), None

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    lib_tag = os.path.basename(nat.LIB_PATH)
    lines = []
    for arm in args.arms.split(","):
        plan, table_bytes = plan_for(arm)
        kwa = dict(kw, goal=plan.goals(B)) if isinstance(plan, kernels.TablePlan) else kw       # each rollout's last table row
        torch.cuda.synchronize()
        ts = []
        res = None
        for i in range(args.reps + 1):                         # the first pass warms up
            flush.fill_(i & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            res = kernels.rollout(plan, B, n_ticks, **kwa)
            b.record()
            torch.cuda.synchronize()
            if i:
                ts.append(a.elapsed_time(b))
        ms = statistics.median(ts)
        read = B * (n_ticks // 10) * 56
        m = res.metrics
        line = {"arm": arm, "rollouts": B, "ticks": n_ticks, "kernel_ms_median": round(ms, 4), "kernel_ms_min": round(min(ts), 4),
                "kernel_ms_all": [round(t, 4) for t in ts], "steps_per_s": B * n_ticks / (ms * 1e-3),
                "table_bytes_resident": table_bytes, "table_bytes_read": read, "table_bytes_per_s": read / (ms * 1e-3),
                "reached_goal": float((m[:, 0] < 0.5).float().mean()), "status_ok": float((m[:, 5] == 0).float().mean()),
                "mean_err_mean": float(m[:, 3].double().mean()), "library": lib_tag, "gpu": name, "power_limit_w": limit,
                "timing": "CUDA events around kernels.rollout, 256 MB L2 flush between passes, median of the timed passes"}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del plan, res
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
