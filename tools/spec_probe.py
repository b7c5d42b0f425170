"""Speculative stretches of K2 (rollout_pair.cuh): CUDA-event timing of the library against variant builds on the bench workload,
alternating, plus the rollback statistics of a counting build -- all in one process, with the card's name and power limit read in
the same run.

    python tools/spec_probe.py [--reps 5] [--variants spec0,h0,h16,u5,u10] [--no-count] [--long] [--out FILE]

Workload: bench.py's K2 launch -- 10^5 lab_course rollouts flown from ONE shared set-point table (10 760 ticks), Monte-Carlo gains /
mass / inertia as bench_workloads.mc_vehicle_arrays draws them, the 4 lab_course boxes, metrics only.  Every timed launch follows a
256 MB L2 flush, as in bench.py.  A round times every library once (its mean over --launches launches); rounds alternate the libraries
--reps times, and each library reports the mean and spread of its rounds.

Libraries: `default` is the package's own build (uav-autonomous-control_b200/lib, built if missing); the variants are build.py
--variant builds of the same sources with the -D flags of VARIANTS (built under build/variants if missing):
  spec0  -DUAVB_SPECULATE=0: every stretch flies the exact body (the kernels of the previous release)
  h0 / h16        UAVB_SPEC_HOLD = 0 / 16 non-watching stretches flown exactly after a rollback (default 4)
  u5 / u10        UAVB_SPEC_UNROLL = 5 / 10 ticks per iteration of the speculative loop (default 2)
  count  -DUAVB_SPEC_COUNT=1 -DUAVB_SPEC_HOLD=0: speculates every non-watching stretch and counts, per warp and stretch (= outer
         period), watching stretches, non-watching ones, rollbacks and which rare path raised them.  Not for timing.
The counting build is run on the bench workload and on the same workload with the wind of BASELINE configs[3] added (+-0.08 N per
axis and rollout, bench_workloads.config3's draw), still flown from one shared table.

Metrics of every library are compared with the default's bit for bit (they must be equal: the speculative body replays exactly).
--long also times BASELINE configs[4]'s per-GPU share (bench_workloads.config4_share) with the default and spec0 libraries.
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

VARIANTS = {
    "spec0": ["-DUAVB_SPECULATE=0"],
    "h0": ["-DUAVB_SPEC_HOLD=0"],
    "h16": ["-DUAVB_SPEC_HOLD=16"],
    "u5": ["-DUAVB_SPEC_UNROLL=5"],
    "u10": ["-DUAVB_SPEC_UNROLL=10"],
    "count": ["-DUAVB_SPEC_COUNT=1", "-DUAVB_SPEC_HOLD=0"],
}
COUNT_NAMES = ("watching", "non_watching", "speculated", "rolled_back", "limit_any", "large_rotation_any")


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


def library_path(tag):
    """Path of a built library (the package's own for 'default'), building it when missing."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("uavb_build", os.path.join(ROOT, "uav-autonomous-control_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    if tag == "default":
        return mod.build()
    path = os.path.join(ROOT, "build", "variants", f"libuavb_{tag}.so")
    return path if os.path.exists(path) else mod.build_variant(tag, VARIANTS[tag])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rollouts", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=3, help="timed launches per library and round")
    ap.add_argument("--variants", default="spec0")
    ap.add_argument("--no-count", action="store_true")
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

    tags = ["default"] + [t for t in args.variants.split(",") if t]
    if not args.no_count:
        tags.append("count")
    libs = {}
    for t in tags:                                     # one CDLL per build; nat._lib selects the one kernels.* calls
        nat._lib, nat.LIB_PATH = None, library_path(t)
        libs[t] = nat.lib()
        libs[t].uavb_dev_speculation.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int]

    def use(t):
        nat._lib = libs[t]

    B = args.rollouts
    use("default")
    plan, kw = wl.lab_course(kernels, dev)
    n_ticks = 10 * int(plan.total_rows.sum())
    mc = wl.mc_vehicle_arrays(kernels, nat, dev, B)
    kw = dict(kw, mc_gains=mc[:11], mc_mass=mc[11], mc_inertia=mc[12:15])
    wind = kernels.mc_uniform(32, B, [-0.08] * 3, [0.08] * 3, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def launch_ms(extra=None):
        ts, res = [], None
        for i in range(args.launches):
            for k in range(8):
                flush.fill_((i + k) & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            res = kernels.rollout(plan, B, n_ticks, **(extra or kw))
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.mean(ts), res.metrics.cpu().numpy()

    header = {"gpu": name, "power_limit_w": limit, "rollouts": B, "ticks": n_ticks, "libraries": {t: os.path.basename(getattr(libs[t], "_name", t)) for t in tags},
              "timing": f"CUDA events around kernels.rollout after a 256 MB L2 flush; a round = mean of {args.launches} launches per library"}
    print(json.dumps(header), flush=True)
    lines = [header]

    timed = [t for t in tags if t != "count"]
    for t in timed:                                    # warm-up: module load of every library
        use(t)
        launch_ms()
    rounds = {t: [] for t in timed}
    outs = {}
    for r in range(args.reps):
        for t in (timed if r % 2 == 0 else timed[::-1]):
            use(t)
            ms, m = launch_ms()
            rounds[t].append(ms)
            outs[t] = m
    ref = outs["default"]
    for t in timed:
        v = rounds[t]
        line = {"library": t, "k2_ms_mean": statistics.mean(v), "k2_ms_stdev": statistics.stdev(v) if len(v) > 1 else 0.0,
                "k2_ms_min": min(v), "k2_ms_max": max(v), "k2_ms_rounds": [round(x, 4) for x in v],
                "metrics_equal_default": bool(np.array_equal(outs[t], ref, equal_nan=True)), "gpu": name, "power_limit_w": limit}
        print(json.dumps(line), flush=True)
        lines.append(line)

    # the exact body forced through the development switch: same metrics
    use("default")
    libs["default"].uavb_dev_speculation(1, None, 0)
    _, m_exact = launch_ms()
    libs["default"].uavb_dev_speculation(0, None, 0)
    line = {"check": "default library with the exact body forced", "metrics_equal_default": bool(np.array_equal(m_exact, ref, equal_nan=True))}
    print(json.dumps(line), flush=True)
    lines.append(line)

    if not args.no_count:
        use("count")
        for label, extra in (("bench", kw), ("bench + wind +-0.08 N", dict(kw, mc_wind=wind))):
            counts = (ctypes.c_ulonglong * 8)()
            libs["count"].uavb_dev_speculation(-1, None, 1)
            saved, args.launches = args.launches, 1
            launch_ms(extra)
            args.launches = saved
            torch.cuda.synchronize()
            libs["count"].uavb_dev_speculation(-1, counts, 0)
            c = dict(zip(COUNT_NAMES, [int(x) for x in counts[:6]]))
            tot = c["watching"] + c["non_watching"]
            nw = max(c["non_watching"], 1)
            line = {"workload": label, "counts_per_warp_stretch": c, "watching_share": c["watching"] / max(tot, 1),
                    "limit_share_of_non_watching": c["limit_any"] / nw, "large_rotation_share_of_non_watching": c["large_rotation_any"] / nw,
                    "rollback_share_of_non_watching": c["rolled_back"] / nw, "note": "counting build, UAVB_SPEC_HOLD=0: every non-watching stretch speculates"}
            print(json.dumps(line), flush=True)
            lines.append(line)

    if args.long:
        use("default")
        fly, _ = wl.config4_share(kernels, nat, dev)
        res = {t: [] for t in ("default", "spec0") if t in libs}
        for t in res:                                  # warm-up
            use(t)
            fly()
            torch.cuda.synchronize()
        for r in range(2):
            for t in res:
                use(t)
                ms, _ = wl.event_ms(fly, reps=1, warm=0)
                res[t].append(ms)
        for t, v in res.items():
            line = {"workload": "long_horizon (BASELINE configs[4] share: 1.25e6 rollouts x 60 000 ticks, 3 chunked launches)", "library": t,
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
