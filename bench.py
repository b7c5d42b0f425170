#!/usr/bin/env python
"""Headline benchmark of the batched closed-loop flight path (BASELINE.json metric: drone-sim-steps/s; min-snap solves/s).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...          # the reference's own classes (oracle/_ref) on the host cores
    python bench.py ... --dump-outputs DIR        # also write the last timed step's per-rollout metrics as DIR/*.npy

Workload (config.workload): BASELINE.json configs[2] -- 10^5 lab_course rollouts per GPU with Monte-Carlo PID gains and
mass/inertia perturbations, velocity 3.0 (config.ini) => 10 760 ticks each, 1.076e9 drone-sim-steps per GPU and step.  One "step" =
one pass of the hot path over the batch: min-snap solve of the mission (K1, take-off + course tables), table geometry, persistent
rollout (K2) of every drone over the whole mission, metrics written.  Consecutive steps are software-pipelined: the planner of step
s + 1 is enqueued on a side stream while K2 of step s flies (K plans per K timed steps, the first one exposed; see hot_path).
Weak scaling: every rank flies its own 10^5 rollouts
(Monte-Carlo inputs keyed by the global rollout index); the per-rollout metrics of a step are all-gathered over NCCL
asynchronously (sharding.MetricGather), overlapping the next step's kernels, and the last gather is inside the timed region.

`value`   : steps/s with inputs resident in HBM (CUDA events around the K timed steps, max over ranks).
`e2e`     : same metric through the reference-facing C-ABI call uavb_fly_mission_host with HOST buffers: per step the waypoints and
            the Monte-Carlo arrays are copied from pinned host memory, the mission is planned and flown, the metrics are copied back
            and the call synchronises.
`roofline`: K2 moves ~0 HBM bytes per tick in metrics-only mode and has no dense contraction (no tensor path): it is bound by the
            SM's register-operand bandwidth (profiles/r02_ffma2_probe.md).  `achieved` = 269 algorithmic flop/tick (DESIGN.md) x
            ticks / K2 time; `peak` = FP32 FMA rate measured in this run (uavb_measure_fma_rates); `peak_three_operand` = the rate
            of FMAs with three distinct register sources measured in the same call; `peak_nominal` = SMs x 128 x 2 x max clock.
`roofline_log`, `solves`, `per_rollout_missions`, `long_horizon`, `sample_table`, `rrt`: the other BASELINE configs and kernels, each
            with its own roofline where one applies; `parity`: the CUDA path against the oracle / the reference's own classes on
            seeded inputs (checker leg, outside every timed region).
`cpu_baseline` / `--impl reference`: the reference's own TrajectoryController + CascadedController + Quad + MinimumSnap objects,
            byte-compiled into oracle/_ref (oracle/build_ref.py), with MuJoCo's rigid-body step restated by oracle/freebody.py --
            kind "reference"; the NumPy port is the fallback (kind "port") when oracle/_ref is absent.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_TICK = 269          # algorithmic flop per drone tick with 4 AABBs: 239 in the 1 kHz body + 298/10 from the 100 Hz loop (DESIGN.md "K2 work per tick")
K2_DRAM_BYTES_PER_LAUNCH = 9.0e6    # ncu: 6.2 MB read + 2.9 MB written per launch of the bench workload (metrics-only: ~0 B per tick; profiles/r02_ncu_rollout_final2.md)
LOG_BYTES_PER_TICK = 52      # 13 fp32 state words (SURVEY 8(d))
ROLLOUTS_PER_GPU = 100_000   # BASELINE configs[2]
VELOCITY = 3.0               # config.ini:7
FREQUENCY = 10               # config.ini:2
TICKS_PER_ROLLOUT = 10_760   # lab_course at v = 3: 1076 table rows x 10 (read back from the plan in the GPU arm)
METRIC = "drone-sim-steps/s"
DUMP_BYTES = 64 << 20        # --dump-outputs budget over all files


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rollouts", type=int, default=ROLLOUTS_PER_GPU, help="rollouts per GPU (default: BASELINE configs[2])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (other configs, K1 / K3 / RRT*, log mode, parity)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="wall-clock budget of the CPU baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed paths returned in their last timed step as DIR/<name>.npy "
                    f"(at most {DUMP_BYTES >> 20} MB in all: a fixed, seeded sample of rows when larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm reports rates only")
    return args


def workload_name(rollouts):
    return (f"BASELINE configs[2]: {rollouts} lab_course rollouts per GPU, Monte-Carlo gains x U(0.8,1.2), mass/inertia x U(0.9,1.1), "
            f"v={VELOCITY} m/s, 10760 ticks each, 4 AABBs, metrics only")


def config_dict(rollouts, n_ticks):
    """`config` of the JSON line -- the same dict in both arms."""
    return {"workload": workload_name(rollouts), "rollouts_per_gpu": rollouts, "ticks_per_rollout": n_ticks, "frequency": FREQUENCY,
            "l2": "256 MB buffer written between timed iterations (L2 flush)", "fp64_parts": "K1 solve and 100 Hz set-point evaluation"}


# ------------------------------------------------------------------------------------------ CPU arm
_TABLE_CACHE = {}


def cpu_kind():
    from oracle import ref_arm
    return "reference" if ref_arm.available() else "port"


def lab_course_table(velocity):
    """(table, waypoints, obstacles) of the lab_course mission: the reference's own _generate_mission_trajectory when oracle/_ref is
    built, else the oracle planner (cached per process)."""
    if velocity not in _TABLE_CACHE:
        from oracle import minsnap_np, ref_arm
        from uav_ac_b200.simulation.scene import LAB_COURSE_OBSTACLES, LAB_COURSE_WAYPOINTS
        if ref_arm.available():
            tab = ref_arm.mission_table(LAB_COURSE_WAYPOINTS, LAB_COURSE_OBSTACLES, velocity, 0.01)
        else:
            tab = minsnap_np.mission_table(LAB_COURSE_WAYPOINTS, LAB_COURSE_OBSTACLES, velocity, 0.01)
        _TABLE_CACHE[velocity] = (tab, LAB_COURSE_WAYPOINTS, LAB_COURSE_OBSTACLES)
    return _TABLE_CACHE[velocity]


def _cpu_worker(job):
    """Fly `missions` whole Monte-Carlo-perturbed lab_course missions (or `ticks` ticks of one when ticks > 0); (ticks, seconds)."""
    seed, missions, ticks = job
    import numpy as np
    from oracle import flight_np, ref_arm
    tab, wp, obs = lab_course_table(VELOCITY)
    total, t0 = 0, time.perf_counter()
    for m in range(max(1, missions)):
        n = ticks if ticks > 0 else FREQUENCY * len(tab)
        if ref_arm.available():
            ref_arm.timed_ticks(seed * 1000 + m, n, tab, wp[0], obs, wp[-1])
        else:
            rng = np.random.default_rng(seed * 1000 + m)
            veh = flight_np.Vehicle().perturbed(rng.uniform(0.8, 1.2, 11), rng.uniform(0.9, 1.1), rng.uniform(0.9, 1.1, 3))
            flight_np.closed_loop(veh, tab, wp[0], obstacles=obs, goal=wp[-1], n_ticks=n)
        total += n
        if ticks > 0:
            break
    return total, time.perf_counter() - t0


def cpu_rollout_rate(seconds: float, cores: int | None = None, pool=None):
    """Whole-machine rate of the reference's Python path (one drone per process, small-array NumPy calls per tick) on a bounded sample
    of the headline workload: every host core flies the same number (>= 1) of WHOLE Monte-Carlo missions.  One estimator for
    `cpu_baseline` and for every step of `--impl reference`."""
    import multiprocessing as mp
    cores = cores or os.cpu_count() or 1
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(cores)
    try:
        probe = pool.map(_cpu_worker, [(i, 0, 300) for i in range(cores)])       # also warms imports and the table
        per_mission = TICKS_PER_ROLLOUT * max(p[1] for p in probe) / 300.0
        missions = max(1, int(seconds / per_mission))
        t0 = time.perf_counter()
        done = pool.map(_cpu_worker, [(1000 + i, missions, 0) for i in range(cores)])
        wall = time.perf_counter() - t0
    finally:
        if own:
            pool.close()
            pool.join()
    total = sum(d[0] for d in done)
    src = "TrajectoryController + CascadedController + Quad of the reference (oracle/_ref) + oracle/freebody.py" if cpu_kind() == "reference" else "oracle/flight_np.py"
    return total / wall, cores, f"{cores} processes x {missions} whole Monte-Carlo lab_course missions of {total // (cores * missions)} ticks (v={VELOCITY}), {src}"


def _solve_worker(job):
    seed, n = job
    import numpy as np
    from oracle import minsnap_np, ref_arm
    rng = np.random.default_rng(seed)
    wp = rng.uniform([2, 2, -5], [22, 12, -1], (n, 5, 3))
    t0 = time.perf_counter()
    for i in range(n):
        if ref_arm.available():
            ref_arm.solve_lstsq(wp[i], 2.5, "lstsq")
        else:
            minsnap_np.solve_coeffs(wp[i], 2.5, "lstsq")
    return n, time.perf_counter() - t0


def cpu_solve_rate(seconds: float = 3.0):
    """MinimumSnap._compute_spline_parameters("lstsq") (minimum_snap.py:138-153, the reference default) on 5-waypoint missions, one process
    per host core (BASELINE.md 3.1)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    with mp.get_context("fork").Pool(cores) as pool:
        probe = pool.map(_solve_worker, [(i, 20) for i in range(cores)])
        per = max(p[1] for p in probe) / 20.0
        n = max(20, int(seconds / per))
        t0 = time.perf_counter()
        done = pool.map(_solve_worker, [(100 + i, n) for i in range(cores)])
        wall = time.perf_counter() - t0
    return {"value": sum(d[0] for d in done) / wall, "unit": "solves/s", "cores": cores, "kind": cpu_kind(),
            "sample": f"{cores} processes x {n} solves of MinimumSnap._compute_spline_parameters('lstsq'), 5 waypoints"}


def cpu_rollout_rate_c(seconds: float):
    """The C twin of the oracle (oracle/oracle_c.c, -O2, one thread per host core) on whole missions: what an optimised scalar CPU
    implementation of the path reaches on this host (reported next to the reference's own figure)."""
    import numpy as np
    from oracle import c_port, flight_np, minsnap_np
    from uav_ac_b200.simulation.scene import LAB_COURSE_OBSTACLES, LAB_COURSE_WAYPOINTS
    cores = os.cpu_count() or 1
    tab = minsnap_np.mission_table(LAB_COURSE_WAYPOINTS, LAB_COURSE_OBSTACLES, VELOCITY, 0.01)
    wp, obs = LAB_COURSE_WAYPOINTS, LAB_COURSE_OBSTACLES
    rng = np.random.default_rng(7)
    def vehicles(n):
        return [flight_np.Vehicle().perturbed(rng.uniform(0.8, 1.2, 11), rng.uniform(0.9, 1.1), rng.uniform(0.9, 1.1, 3)) for _ in range(n)]
    t0 = time.perf_counter()
    c_port.closed_loop_batch(vehicles(cores), tab, wp[0], obstacles=obs, goal=wp[-1], threads=cores)
    per = max(time.perf_counter() - t0, 1e-4)                      # one full mission per core
    n = max(cores, min(4096, int(cores * seconds / per)))
    vs = vehicles(n)
    t0 = time.perf_counter()
    c_port.closed_loop_batch(vs, tab, wp[0], obstacles=obs, goal=wp[-1], threads=cores)
    wall = time.perf_counter() - t0
    return n * FREQUENCY * len(tab) / wall, cores, f"{n} whole Monte-Carlo lab_course missions (v={VELOCITY}) on {cores} threads, oracle/oracle_c.c"


def run_reference(args):
    """--impl reference: the reference's own classes (oracle/_ref; fallback: the oracle port) on all host cores.  A step is a bounded
    sample of the workload -- one whole Monte-Carlo mission per host core -- and ms_per_step is extrapolated to the full batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    vals, sample = [], ""
    with mp.get_context("fork").Pool(cores) as pool:
        for i in range(args.warmup + args.steps):
            v, cores, sample = cpu_rollout_rate(1.0, cores, pool)              # 1 s budget => exactly one whole mission per core
            if i >= args.warmup:
                vals.append(v)
    value = statistics.mean(vals)
    ms = 1e3 * args.rollouts * TICKS_PER_ROLLOUT / value
    line = {
        "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "impl": "reference",
        "config": config_dict(args.rollouts, TICKS_PER_ROLLOUT),
        "note": "each step is a bounded sample (one whole mission per host core); ms_per_step is extrapolated to the full batch",
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": cpu_kind(), "sample": sample},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).

    A thread polls NVML (nvidia-ml-py) every ~2 ms -- the timed region of the default run lasts tens of
    milliseconds, too short for `nvidia-smi -lms`; nvidia-smi is the fallback when NVML cannot be loaded."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
               "hw_power_brake_slowdown": 0x80}

    def __init__(self, index):
        import threading
        self.index, self.samples, self.stop_flag, self.thread = index, [], threading.Event(), None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(local):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local < len(ids) and ids[local].isdigit():
                return int(ids[local])
        return local

    def _poll(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                try:
                    why = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    why = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                self.samples.append((sm, why, pw))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        import threading
        if self.nvml is None:
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def stop(self):
        if self.nvml is None:
            return self._smi_once()
        self.stop_flag.set()
        self.thread.join(timeout=2)
        if not self.samples:
            return self._smi_once()
        reasons = set()
        for _, why, _ in self.samples:
            for name, bit in self.REASONS.items():
                if why & bit:
                    reasons.add(name)
        return {"sm_mhz": statistics.median(s[0] for s in self.samples), "sm_max_mhz": float(self.max_sm), "reasons": sorted(reasons),
                "power_w_max": max(s[2] for s in self.samples), "samples": len(self.samples), "source": "nvml, 2 ms poll during the timed region"}

    def _smi_once(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                 capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0]
            p = [x.strip() for x in out.split(",")]
            reasons = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]) if v.lower().startswith("active")]
            return {"sm_mhz": float(p[0]), "sm_max_mhz": float(p[1]), "reasons": reasons, "power_w_max": float(p[2]), "samples": 1,
                    "source": "nvidia-smi, one sample right after the timed region (NVML unavailable)"}
        except Exception as e:  # noqa: BLE001
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"clock sampling unavailable: {e}"]}


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import bench_workloads as wl
    from uav_ac_b200 import _native as nat, host_api, kernels, sharding
    from uav_ac_b200.simulation.scene import LAB_COURSE_GOAL, LAB_COURSE_OBSTACLES, LAB_COURSE_START, LAB_COURSE_WAYPOINTS

    rank, local, world = sharding.init_from_env("nccl")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    nat.lib()
    B = args.rollouts
    total = B * world
    begin, end = sharding.shard_range(total, rank, world)
    assert end - begin == B

    # ---- host inputs (pinned): waypoints, velocity, Monte-Carlo scales as a user would hand them over
    veh = nat.default_vehicle()
    mc_dev = wl.mc_vehicle_arrays(kernels, nat, dev, B, index_base=begin)                   # [15, B] fp32, keyed by the global rollout index
    mc_host = mc_dev.cpu().pin_memory()
    wp_host = torch.tensor(LAB_COURSE_WAYPOINTS, dtype=torch.float64).pin_memory()
    vel_host = torch.tensor([VELOCITY], dtype=torch.float64).pin_memory()
    obs = torch.tensor(LAB_COURSE_OBSTACLES, dtype=torch.float32, device=dev)
    obs64 = torch.tensor(LAB_COURSE_OBSTACLES, dtype=torch.float64, device=dev)
    start = torch.tensor(LAB_COURSE_START, dtype=torch.float64, device=dev)
    goal = torch.tensor(LAB_COURSE_GOAL, dtype=torch.float64, device=dev)
    metrics_host = torch.empty((B, nat.N_METRICS), dtype=torch.float32).pin_memory()
    wp_dev = wp_host.to(dev)
    vel_dev = vel_host.to(dev)
    gather = sharding.MetricGather(B, nat.N_METRICS, total, dev)
    results = [kernels.RolloutResult(gather.shard[i], None, None, None) for i in range(2)]
    state = {"n": None, "k": 0, "plans": []}

    side = torch.cuda.Stream(dev)                            # the NEXT step's plan is enqueued here while this step's K2 flies
    state.update(pending=None, remaining=0)

    def make_plan(wp, vel, n_ticks):
        return kernels.plan_missions([(wp[None, :2].contiguous(), vel), (wp[None, 1:].contiguous(), vel)], FREQUENCY * veh.dt, shared=True,
                                     table_rows=None if n_ticks is None else n_ticks // FREQUENCY, obstacles=obs64)

    def issue_plan(wp, vel, mark):
        """A speculative plan on the side stream, ordered behind `mark` -- the point of the launching stream at which the step that
        issues it began, so the plan belongs to that step's timed bracket but does not wait for the step's K2 --, with the event the
        K2 that flies it waits for."""
        side.wait_event(mark)
        with torch.cuda.stream(side):
            plan = make_plan(wp, vel, state["n"])
            ready = torch.cuda.Event()
            ready.record(side)
        state["plans"].append(plan)                          # speculative plan (no host round trip): its report is checked in drain()
        return plan, ready

    def hot_path(wp, vel, mc, result):
        """Plan (both tables through K1 and the obstacle-correction sweep, table geometry, set-point table) + K2 over the shard; the
        per-rollout metrics land in result.metrics.  After the first step the table length is known and the plan is speculative
        (kernels.plan_missions: no host round trip, the correction loop's report is verified in drain(), inside the timed region).
        Steps are software-pipelined: the plan of step s + 1 is enqueued on a side stream behind the LAUNCH of K2(s) -- its few small
        kernels run in the SM slots K2(s) frees at its tail -- and K2(s + 1) waits for its event.  The first step of a timed
        region plans inside the region (drain() drops a plan made ahead), the last one plans nothing ahead: K plans per K steps."""
        main = torch.cuda.current_stream(dev)
        mark = torch.cuda.Event()
        mark.record(main)                                    # this step begins here on the launching stream
        if state["n"] is None:                               # mission length is data dependent: read it once, outside the timed steps
            plan = make_plan(wp, vel, None)
            state["n"] = FREQUENCY * int(plan.total_rows.item())
        else:
            plan, ready = state["pending"] if state["pending"] is not None else issue_plan(wp, vel, mark)
            state["pending"] = None
            main.wait_event(ready)
        kernels.rollout(plan, B, state["n"], start=start, goal=goal, vehicle=veh, frequency=FREQUENCY, mc_gains=mc[:11], mc_mass=mc[11],
                        mc_inertia=mc[12:15], obstacles=obs, want_state=False, out=result, index_base=begin)
        state["remaining"] -= 1
        if state["remaining"] > 0:
            state["pending"] = issue_plan(wp, vel, mark)

    def step_device():
        k = state["k"]
        gather.local(k)                                      # orders this step's K2 after the gather that last read the same shard buffer
        hot_path(wp_dev, vel_dev, mc_dev, results[k % 2])
        gather.launch(k)                                     # asynchronous: overlaps the next step's K1 / K2
        state["k"] = k + 1

    def drain():
        if state["k"]:
            gather.result(state["k"] - 1)                    # the last gather belongs to the timed region
        for plan in state["plans"]:                          # every speculative plan of the region is the plan the reference makes
            plan.verify()
        state["plans"].clear()
        state["pending"] = None

    mc_mass_h, mc_inertia_h, mc_gains_h = mc_host[11], mc_host[12:15], mc_host[:11]     # contiguous pinned views, SoA
    wp_np = np.ascontiguousarray(LAB_COURSE_WAYPOINTS, dtype=np.float64)

    def step_e2e():
        """The reference-facing call: uavb_fly_mission_host (C ABI, HOST buffers).  Inside the call: H2D of the
        waypoints and the Monte-Carlo arrays, K1 x2, table geometry, K2, D2H of the metrics, synchronisation."""
        host_api.fly_mission_host(wp_np, VELOCITY, B, n_takeoff_waypoints=2, frequency=FREQUENCY, vehicle=veh, mc_mass=mc_mass_h,
                                  mc_inertia=mc_inertia_h, mc_gains=mc_gains_h, obstacles=LAB_COURSE_OBSTACLES, start=LAB_COURSE_START,
                                  goal=LAB_COURSE_GOAL, metrics_out=metrics_host)

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)                    # > 126 MB L2

    def timed(fn, steps, warmup, sampler=None, wall=False, after=None):
        """K timed steps between barriers + synchronize; device time from CUDA events on the launching (current torch)
        stream, or host wall-clock for the synchronous host-buffer call (wall=True); max over ranks."""
        state["remaining"] = warmup
        for _ in range(warmup):
            fn()
        if after:
            after()
        state["remaining"] = steps
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        wall_ms = 0.0
        for s in range(steps):
            if s == 0 and not wall:
                flush_and_space(flush, 0)                                                   # L2 flush + ~0.3 ms of queued work: the first step's launches are enqueued before the GPU reaches them
            else:
                flush.fill_(s & 0xFF)                                                       # flush L2 between timed iterations
            if wall:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                wall_ms += (time.perf_counter() - t0) * 1e3
            else:
                ev[s][0].record()
                fn()
                if after and s == steps - 1:
                    after()
                ev[s][1].record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms = wall_ms if wall else sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), clocks

    W = max(args.warmup, 3)
    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev, clocks = timed(step_device, args.steps, W, sampler, after=drain)
    dumped = {"metrics": gather.result(state["k"] - 1).cpu().numpy()} if args.dump_outputs and rank == 0 else None    # [total, 8] fp32
    n_ticks = state["n"]
    ms_e2e, _ = timed(step_e2e, args.steps, 2, wall=True)
    torch.cuda.synchronize()
    if dumped is not None:
        dumped["e2e_metrics"] = metrics_host.numpy()                                         # this rank's [B, 8] fp32
        dump_outputs(args.dump_outputs, dumped)
    sim_steps = float(total) * n_ticks                                                       # whole job, one step
    value = sim_steps * args.steps / (ms_dev * 1e-3)
    e2e = sim_steps * args.steps / (ms_e2e * 1e-3)
    last = results[(state["k"] - 1) % 2]

    # ---- K2 alone: average launch duration with events on the launching stream
    plan = kernels.plan_missions([(wp_dev[None, :2].contiguous(), vel_dev), (wp_dev[None, 1:].contiguous(), vel_dev)], FREQUENCY * veh.dt, shared=True)
    kw = dict(start=start, goal=goal, vehicle=veh, frequency=FREQUENCY, mc_gains=mc_dev[:11], mc_mass=mc_dev[11], mc_inertia=mc_dev[12:15],
              obstacles=obs, want_state=False, out=last)
    k2 = []
    for i in range(2 + args.steps):
        flush_and_space(flush, i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); kernels.rollout(plan, B, n_ticks, **kw); b.record()
        torch.cuda.synchronize()
        if i >= 2:
            k2.append(a.elapsed_time(b))
    k2_ms = statistics.mean(k2)
    # per-rank K2 time: the skew the max-over-ranks timing pays for
    k2_all = torch.tensor([k2_ms], dtype=torch.float64, device=dev)
    if world > 1:
        k2_list = [torch.zeros_like(k2_all) for _ in range(world)]
        dist.all_gather(k2_list, k2_all)
        k2_ranks = [float(x.item()) for x in k2_list]
    else:
        k2_ranks = [k2_ms]
    summary = sharding.summarize(last.metrics)

    # ---- the north-star job shape under torchrun: every rank flies one GPU's share of configs[4] (10^7 x 60 s over 8 GPUs), metrics gathered
    long_h = None
    if not args.no_extras:
        long_h = long_horizon(wl, kernels, nat, sharding, dev, rank, world, dist)

    line = None
    if rank == 0:
        fp32_peak, fp32_peak3, fp64_peak = nat.measure_fma_rates(local)
        sms = nat.device_info(local)[0]
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        sm_max = (clocks or {}).get("sm_max_mhz") or peaks.get("sm_max_mhz") or 1965.0
        achieved = FLOP_PER_TICK * float(B) * n_ticks / (k2_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": config_dict(B, n_ticks),
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "steps/s", "h2d_bytes_per_step": int(mc_host.numel() * 4 + wp_host.numel() * 8 + 8),
                    "d2h_bytes_per_step": int(metrics_host.numel() * 4), "ms_per_step": ms_e2e / args.steps,
                    "call": "uavb_fly_mission_host (C ABI, pinned host buffers, synchronous); host wall-clock, max over ranks"},
            # own kernels per step (torch glue not counted): correct_classify, minsnap_solve_list x2 (take-off: <= 4 splines, course: <= 8),
            # correct_sweep (one launch for every bucket), minsnap_pack, table_meta_warp, shared_seg_flags, target_rows, target_heading,
            # rollout_sliced -- the ncu launch list of the same command counts the same ten (profiles/r02_launches_final2.md)
            "gpu_launches": 10 * args.steps,
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak if fp32_peak else None,
                         "traffic": K2_DRAM_BYTES_PER_LAUNCH, "traffic_unit": "bytes per launch, dram read+write (ncu --set full, profiles/r02_ncu_rollout_final2.md)",
                         "kernel": "rollout_sliced_kernel<MC,TABLE> (two drones per thread, packed fp32x2)", "kernel_ms": k2_ms, "flop_per_tick": FLOP_PER_TICK,
                         "peak_source": "uavb_measure_fma_rates in this run (MEASURED_PEAKS.json carries no fp32 figure)",
                         "peak_three_operand": fp32_peak3, "frac_of_three_operand_peak": achieved / fp32_peak3 if fp32_peak3 else None,
                         "peak_nominal": sms * 128 * 2 * sm_max * 1e6 / 1e12,
                         "limit": "register-operand bandwidth: a scheduler reads two register words per cycle, so FMAs with three distinct register "
                                  "sources run at peak_three_operand (profiles/r02_ffma2_probe.md); frac is against the FMA peak with reuse-cached operands",
                         "fp64_peak_tflops": fp64_peak, "ticks_per_s_k2": float(B) * n_ticks / (k2_ms * 1e-3),
                         "k2_ms_per_rank": k2_ranks},
            "mission_report": summary,
        }
        if long_h is not None:
            line["long_horizon"] = long_h
        if not args.no_extras:
            line["roofline_log"] = log_mode_roofline(kernels, plan, kw, dev, n_ticks, peaks, flush)
            line["solves"] = solve_rate(kernels, host_api, dev, flush, peaks)
            if world == 1:
                for name, fn in (("per_rollout_missions", lambda: per_rollout_missions(wl, kernels, dev, fp32_peak, fp32_peak3)),
                                 ("sample_table", lambda: wl.sample_table_rate(kernels, dev, peaks)), ("rrt", lambda: wl.rrt_rate(dev)),
                                 ("correction_loop", lambda: wl.correction_rate(kernels, nat, dev)),
                                 ("parity", lambda: wl.parity_block(kernels, nat, dev))):
                    try:
                        line[name] = fn()
                    except Exception as e:  # noqa: BLE001  (a side measurement must not take the headline down)
                        line[name] = {"error": f"{type(e).__name__}: {e}"}
    if world > 1:
        dist.barrier()
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            v, cores, sample = cpu_rollout_rate(args.cpu_seconds)
            line["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": cores, "kind": cpu_kind(), "sample": sample}
            if "solves" in line:
                try:
                    line["solves"]["cpu_baseline"] = cpu_solve_rate()
                except Exception as e:  # noqa: BLE001
                    line["solves"]["cpu_baseline"] = {"unavailable": str(e)}
            try:
                vc, cc, sc = cpu_rollout_rate_c(min(args.cpu_seconds, 8.0))
                line["cpu_baseline_c"] = {"value": vc, "unit": "steps/s", "cores": cc, "kind": "port", "sample": sc,
                                          "note": "optimised C restatement; the reference itself is Python/NumPy (cpu_baseline)"}
            except Exception as e:  # noqa: BLE001  (no C compiler on the box: the reference figure stands alone)
                line["cpu_baseline_c"] = {"unavailable": str(e)}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def flush_and_space(flush, i):
    """L2 flush (256 MB written) repeated a few times: besides evicting L2 it keeps the GPU busy for ~0.3 ms, so the host has
    enqueued the start event, the launch and the stop event before the GPU reaches them -- the event pair then brackets the
    kernel(s) of the call, not the host's launch latency (which matters for the sub-millisecond kernels)."""
    for k in range(8):
        flush.fill_((i + k) & 0xFF)


def long_horizon(wl, kernels, nat, sharding, dev, rank, world, dist):
    """BASELINE configs[4] in the north-star job shape: every rank flies ONE GPU's share of 10^7 x 60 s x 1 kHz (1.25e6 rollouts x
    60 000 ticks, three chunked launches through the carry block) and the [B, 8] metrics are all-gathered; at N = 8 this is the whole
    job.  Device time (events), max over ranks, gather included."""
    import torch
    B, ticks = 1_250_000, 60_000
    lo = rank * B
    fly, _ = wl.config4_share(kernels, nat, dev, B=B, ticks=ticks, index_base=lo)
    fly()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    res = fly()
    m = sharding.gather_metrics(res.metrics, B * world) if world > 1 else res.metrics
    b.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    if rank != 0:
        return None
    return {"workload": f"BASELINE configs[4] share: {B} lab_course rollouts per GPU x {ticks} ticks (60 s at 1 kHz), Monte-Carlo vehicles, metrics only, "
                        f"3 chunked launches + metric all-gather; {world} GPU(s) = {B * world} rollouts",
            "rollouts_total": B * world, "ticks": ticks, "ms": ms, "value": float(B) * world * ticks / (ms * 1e-3), "unit": "steps/s",
            "periods_ok": bool((m[:, 7] == ticks // FREQUENCY).all()), "hover_final_dist_max": float(m[:, 0].max()), **sharding.summarize(m)}


def per_rollout_missions(wl, kernels, dev, fp32_peak, fp32_peak3):
    """BASELINE configs[3] at full size: 10^6 rollouts, per-rollout missions (on-the-fly fp64 set-points), wind, 64 sets x 6 AABBs."""
    import torch
    B = 1_000_000
    fly, n_ticks, info = wl.config3(kernels, dev, B=B)
    res = kernels.RolloutResult(torch.empty((B, 8), dtype=torch.float32, device=dev), None, None, None)
    ms, _ = wl.event_ms(lambda: fly(res), reps=2, warm=1)
    m = res.metrics
    achieved = FLOP_PER_TICK * float(B) * n_ticks / (ms * 1e-3) / 1e12
    return {"workload": f"BASELINE configs[3]: {B} rollouts, random 5-waypoint missions (take-off + course), wind +-0.08 N, 64 obstacle sets x 6 AABBs, metrics only",
            "value": float(B) * n_ticks / (ms * 1e-3), "unit": "steps/s", "rollouts": B, "ticks": n_ticks, "kernel_ms": ms,
            "collision_fraction": float((m[:, 1] > 0).float().mean()), "failed_fraction": float((m[:, 5] != 0).float().mean()),
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak if fp32_peak else None,
                         "peak_three_operand": fp32_peak3, "flop_per_tick": FLOP_PER_TICK, "kernel": "rollout_sliced_scalar_kernel<MC> (one drone per thread, on-the-fly set-points)", "traffic": None}}


def log_mode_roofline(kernels, plan, kw, dev, n_ticks, peaks, flush):
    """Full-rate state log (52 B/tick): HBM roofline of the logging epilogue (north_star)."""
    import torch
    Bl = 151552                                           # two full waves of 148 SMs x 8 CTAs x 64 drones
    ticks = 400                                           # 151552 x 400 x 52 B = 3.15 GB of log per launch
    from uav_ac_b200 import _native as nat
    import bench_workloads as wl
    kw = dict(kw)
    mc = wl.mc_vehicle_arrays(kernels, nat, dev, Bl)
    kw.update(mc_gains=mc[:11], mc_mass=mc[11], mc_inertia=mc[12:15])
    kw["out"] = None
    kw["want_metrics"] = False
    log = torch.empty((ticks, 13, Bl), dtype=torch.float32, device=dev)
    res = kernels.RolloutResult(None, None, log, None)
    kw["out"] = res
    ms = []
    for i in range(4):
        flush_and_space(flush, i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); kernels.rollout(plan, Bl, ticks, log_stride=1, **kw); b.record()
        torch.cuda.synchronize()
        if i >= 1:
            ms.append(a.elapsed_time(b))
    t = statistics.mean(ms) * 1e-3
    gbs = LOG_BYTES_PER_TICK * float(Bl) * ticks / t / 1e9
    peak = peaks.get("hbm_gbs", 6650.0)
    return {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "traffic": 3.18e9, "traffic_unit": "bytes per launch, dram read+write (ncu --set full, profiles/r01_ncu_rollout_log_v2.md)",
            "kernel": "rollout_sliced_kernel<MC,TABLE,LOG>", "kernel_ms": t * 1e3, "ticks_per_s": float(Bl) * ticks / t,
            "rollouts": Bl, "ticks": ticks,
            "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)",
            "note": "full-rate state log: rollouts x ticks x 52 B written per launch (write-only traffic against the read+write copy peak)"}


def solve_rate(kernels, host_api, dev, flush, peaks):
    """BASELINE configs[1]: 10^6 random 5-waypoint missions -- K1 with inputs resident in HBM, and end to end through the host-buffer
    call uavb_minsnap_solve_f64_host (pinned host buffers in and out)."""
    import torch
    Bm = 1_000_000
    wp, vel = kernels.mc_missions(99, Bm, 4, device=dev)
    ms = []
    for i in range(6):
        flush_and_space(flush, i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); kernels.minsnap_solve(wp, vel); b.record()
        torch.cuda.synchronize()
        if i >= 2:
            ms.append(a.elapsed_time(b))
    t = statistics.mean(ms) * 1e-3
    byts = 928.0 * Bm                                      # 128 B in + 800 B out per solve (SURVEY 8(d))
    peak = peaks.get("hbm_gbs", 6650.0)
    out = {"metric": "min-snap solves/s", "value": Bm / t, "unit": "solves/s", "missions": Bm, "splines": 4, "kernel_ms": t * 1e3,
           "roofline": {"bound": "hbm", "achieved": byts / t / 1e9, "peak": peak, "unit": "GB/s", "frac": byts / t / 1e9 / peak,
                        "traffic": 8.78e8 * Bm / 1e6, "traffic_unit": "bytes per launch, dram read+write (ncu --set full, profiles/r02_ncu_minsnap_final.md: 130 MB read + 748 MB written per 1e6 solves)",
                        "kernel": "minsnap_solve_stream_kernel<4,4> (persistent, bulk-load prefetch, two staging tiles, tensor stores)",
                        "note": "includes output allocation by torch (cached allocator)"}}
    if hasattr(host_api, "minsnap_solve_host"):
        wp_h, vel_h = wp.cpu().pin_memory(), vel.cpu().pin_memory()
        c_h = torch.empty((Bm, 32, 3), dtype=torch.float64).pin_memory()
        t_h = torch.empty((Bm, 4), dtype=torch.float64).pin_memory()
        s_h = torch.empty((Bm,), dtype=torch.int32).pin_memory()
        ws = []
        for i in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host_api.minsnap_solve_host(wp_h, vel_h, coeffs_out=c_h, times_out=t_h, status_out=s_h)
            if i >= 2:
                ws.append(time.perf_counter() - t0)
        te = statistics.mean(ws)
        h2d, d2h = Bm * 128, Bm * 804
        out["e2e"] = {"value": Bm / te, "unit": "solves/s", "ms": te * 1e3, "h2d_bytes": h2d, "d2h_bytes": d2h,
                      "call": "uavb_minsnap_solve_f64_host (C ABI, pinned host buffers, chunked H2D -> K1 -> D2H pipeline, synchronous)",
                      "link_GBps": (h2d + d2h) / te / 1e9, "note": "bound by the host link: 932 B cross PCIe per solve, 804 of them device-to-host"}
    return out


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy.  An array larger than its share of DUMP_BYTES is cut to a fixed, seeded,
    sorted sample of its rows, the same for every run with the same arguments, so two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096                                                # room for the .npy header
    for name, a in arrays.items():
        if a.nbytes > share:
            keep = share // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, written to the process's original stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    a = parse()
    # Libraries (NCCL's version banner, torchrun warnings) may print to stdout; the contract is ONE JSON line there.
    # Everything else is sent to stderr for the lifetime of the run.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
