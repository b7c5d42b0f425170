"""Speculative stretches of K2 (rollout_pair.cuh): CUDA-event timing of the library on the bench workload, and its metrics with the
exact body forced through uavb_dev_speculation compared bit for bit -- in one process, with the card's name and power limit read in
the same run.

    python tools/spec_probe.py [--reps 5] [--long] [--out FILE]

Workload: bench.py's K2 launch -- 10^5 lab_course rollouts flown from ONE shared set-point table (10 760 ticks), Monte-Carlo gains /
mass / inertia as bench_workloads.mc_vehicle_arrays draws them, the 4 lab_course boxes, metrics only.  Every timed launch follows a
256 MB L2 flush, as in bench.py.  A round is the mean over --launches launches; the library reports the mean and spread of --reps
rounds.  The library is the package's own build (uav-autonomous-control_b200/lib, built if missing).

--long also times BASELINE configs[4]'s per-GPU share (bench_workloads.config4_share).
"""
from __future__ import annotations

import argparse
import ctypes
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
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                             text=True, timeout=20).stdout.strip()
        limit = float(out.splitlines()[0])
    except Exception:                                  # noqa: BLE001 -- reported as unknown, never guessed
        limit = None
    return name, limit


def library_path():
    """Path of the package's own library, building it when missing."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("uavb_build", os.path.join(ROOT, "uav-autonomous-control_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rollouts", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=3, help="timed launches per round")
    ap.add_argument("--long", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import bench_workloads as wl
    from uav_ac_b200 import _native as nat
    from uav_ac_b200 import kernels
    if not torch.cuda.is_available():
        raise SystemExit("spec_probe: no CUDA device (a timing needs the GPU)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, limit = card()

    nat._lib, nat.LIB_PATH = None, library_path()
    lib = nat.lib()
    lib.uavb_dev_speculation.argtypes = [ctypes.c_int]

    B = args.rollouts
    plan, kw = wl.lab_course(kernels, dev)
    n_ticks = 10 * int(plan.total_rows.sum())
    mc = wl.mc_vehicle_arrays(kernels, nat, dev, B)
    kw = dict(kw, mc_gains=mc[:11], mc_mass=mc[11], mc_inertia=mc[12:15])
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def launch_ms():
        ts, res = [], None
        for i in range(args.launches):
            for k in range(8):
                flush.fill_((i + k) & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            res = kernels.rollout(plan, B, n_ticks, **kw)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.mean(ts), res.metrics.cpu().numpy()

    header = {"gpu": name, "power_limit_w": limit, "rollouts": B, "ticks": n_ticks, "library": nat.LIB_PATH,
              "timing": f"CUDA events around kernels.rollout after a 256 MB L2 flush; a round = mean of {args.launches} launches"}
    print(json.dumps(header), flush=True)
    lines = [header]

    launch_ms()                                        # warm-up: module load
    rounds, ref = [], None
    for _ in range(args.reps):
        ms, ref = launch_ms()
        rounds.append(ms)
    line = {"k2_ms_mean": statistics.mean(rounds), "k2_ms_stdev": statistics.stdev(rounds) if len(rounds) > 1 else 0.0,
            "k2_ms_min": min(rounds), "k2_ms_max": max(rounds), "k2_ms_rounds": [round(x, 4) for x in rounds], "gpu": name, "power_limit_w": limit}
    print(json.dumps(line), flush=True)
    lines.append(line)

    # the exact body forced through the development switch: same metrics
    lib.uavb_dev_speculation(1)
    _, m_exact = launch_ms()
    lib.uavb_dev_speculation(0)
    line = {"check": "exact body forced", "metrics_equal_speculative": bool(np.array_equal(m_exact, ref, equal_nan=True))}
    print(json.dumps(line), flush=True)
    lines.append(line)

    if args.long:
        fly, _ = wl.config4_share(kernels, nat, dev)
        fly()                                          # warm-up
        torch.cuda.synchronize()
        v = [wl.event_ms(fly, reps=1, warm=0)[0] for _ in range(2)]
        line = {"workload": "long_horizon (BASELINE configs[4] share: 1.25e6 rollouts x 60 000 ticks, 3 chunked launches)",
                "ms": [round(x, 2) for x in v], "gpu": name, "power_limit_w": limit}
        print(json.dumps(line), flush=True)
        lines.append(line)

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
