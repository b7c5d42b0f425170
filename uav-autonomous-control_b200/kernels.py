"""Tensor-level entry points over the C ABI: batched min-snap solve (K1), table geometry, sampled
tables (K3), mission packing and the persistent closed-loop rollout (K2).

Every function takes/returns CUDA tensors and enqueues on the current torch stream; nothing here
computes on the CPU.  Reference call sites replaced are cited per function (paths relative to
/root/reference).
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import Optional, Sequence

import torch

from . import _native as nat

START_END_TIME_FACTOR = 1.5  # MinimumSnap.START_END_TIME_FACTOR (uav_ac/planning/minimum_snap.py:10)


def _dev(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise nat.UavbError("no CUDA device visible: the batched flight path has no CPU implementation")
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


# ------------------------------------------------------------------------------------------ K1
def minsnap_solve(waypoints: torch.Tensor, velocity: torch.Tensor, factor: float = START_END_TIME_FACTOR):
    """Batched MinimumSnap._compute_spline_parameters (minimum_snap.py:138-153).

    waypoints [B, S+1, 3] f64, velocity [B] f64 -> coeffs [B, 8S, 3], times [B, S], status [B] i32.
    """
    if waypoints.dim() != 3 or waypoints.shape[2] != 3 or waypoints.shape[1] < 2:
        raise ValueError("waypoints must have shape (B, S+1, 3) with S >= 1")
    B, S = waypoints.shape[0], waypoints.shape[1] - 1
    if velocity.shape != (B,):
        raise ValueError("velocity must have shape (B,)")
    dev = waypoints.device
    coeffs = torch.empty((B, 8 * S, 3), dtype=torch.float64, device=dev)
    times = torch.empty((B, S), dtype=torch.float64, device=dev)
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    nat.on(dev).uavb_minsnap_solve_f64(
        nat.ptr(waypoints, torch.float64, "waypoints"), nat.ptr(velocity, torch.float64, "velocity"), B, S, float(factor),
        nat.ptr(coeffs), nat.ptr(times), nat.ptr(status), nat.stream_ptr(dev))
    return coeffs, times, status


def minsnap_solve_ragged(waypoints: torch.Tensor, wp_offsets: torch.Tensor, velocity: torch.Tensor,
                         factor: float = START_END_TIME_FACTOR):
    """Ragged K1: packed waypoints [n_wp, 3], wp_offsets [B+1] i32 -> coeffs [n_seg, 8, 3], times [n_seg], status [B]."""
    B = wp_offsets.numel() - 1
    n_seg = waypoints.shape[0] - B
    dev = waypoints.device
    coeffs = torch.empty((n_seg, 8, 3), dtype=torch.float64, device=dev)
    times = torch.empty((n_seg,), dtype=torch.float64, device=dev)
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    nat.on(dev).uavb_minsnap_solve_ragged_f64(
        nat.ptr(waypoints, torch.float64, "waypoints"), nat.ptr(wp_offsets, torch.int32, "wp_offsets"),
        nat.ptr(velocity, torch.float64, "velocity"), B, float(factor), nat.ptr(coeffs), nat.ptr(times), nat.ptr(status),
        nat.stream_ptr(dev))
    return coeffs, times, status


def minsnap_constraints(waypoints: torch.Tensor, times: torch.Tensor):
    """MinimumSnap.A / MinimumSnap.b of the reference (minimum_snap.py:171-255, same row order) for B missions of S splines:
    waypoints [B, S+1, 3], times [B, S] -> A [B, 6S+2, 8S], b [B, 6S+2, 3]."""
    B, S = waypoints.shape[0], waypoints.shape[1] - 1
    A = torch.empty((B, 6 * S + 2, 8 * S), dtype=torch.float64, device=waypoints.device)
    b = torch.empty((B, 6 * S + 2, 3), dtype=torch.float64, device=waypoints.device)
    nat.on(waypoints.device).uavb_minsnap_constraints_f64(nat.ptr(waypoints, torch.float64, "waypoints"), nat.ptr(times, torch.float64, "times"), B, S,
                                                     nat.ptr(A), nat.ptr(b), nat.stream_ptr(waypoints.device))
    return A, b


def table_meta(coeffs: torch.Tensor, times: torch.Tensor, seg_offsets: torch.Tensor, dt: float):
    """Rows per segment, look-ahead yaw and total rows per table (minimum_snap.py:104, 126-136).

    coeffs [n_seg, 8, 3] (or any contiguous view with 24 doubles per segment), times [n_seg],
    seg_offsets [B+1] i32 -> rows [n_seg] i32, yaw0 [B] f64, total_rows [B] i32.
    """
    B = seg_offsets.numel() - 1
    n_seg = times.numel()
    dev = coeffs.device
    rows = torch.empty((n_seg,), dtype=torch.int32, device=dev)
    yaw0 = torch.empty((B,), dtype=torch.float64, device=dev)
    total = torch.empty((B,), dtype=torch.int32, device=dev)
    nat.on(dev).uavb_minsnap_table_meta_f64(
        nat.ptr(coeffs, torch.float64, "coeffs"), nat.ptr(times, torch.float64, "times"), nat.ptr(seg_offsets, torch.int32, "seg_offsets"),
        B, float(dt), nat.ptr(rows), nat.ptr(yaw0), nat.ptr(total), nat.stream_ptr(dev))
    return rows, yaw0, total


def minsnap_sample(coeffs: torch.Tensor, times: torch.Tensor, seg_offsets: torch.Tensor, seg_rows: torch.Tensor,
                   row_offsets: torch.Tensor, dt: float) -> torch.Tensor:
    """K3: the (N, 11) tables of MinimumSnap._generate_trajectory (minimum_snap.py:97-124), packed over missions."""
    B = seg_offsets.numel() - 1
    n_rows = int(row_offsets[-1].item())
    table = torch.empty((n_rows, 11), dtype=torch.float64, device=coeffs.device)
    nat.on(coeffs.device).uavb_minsnap_sample_f64(
        nat.ptr(coeffs, torch.float64, "coeffs"), nat.ptr(times, torch.float64, "times"), nat.ptr(seg_offsets, torch.int32, "seg_offsets"),
        nat.ptr(seg_rows, torch.int32, "seg_rows"), nat.ptr(row_offsets, torch.int32, "row_offsets"), B, float(dt), nat.ptr(table),
        nat.stream_ptr(coeffs.device))
    return table


def table_hits(table: torch.Tensor, row_offsets: torch.Tensor, cuboid: torch.Tensor, hit_mask: torch.Tensor) -> torch.Tensor:
    """OR into hit_mask [B] (int64 bit s) the splines with a sampled point inside `cuboid` ([6] or [B, 6])
    -- the test of the correction loop (minimum_snap.py:84-87, 327-357)."""
    B = row_offsets.numel() - 1
    stride = 0 if cuboid.dim() == 1 else 6
    nat.on(table.device).uavb_minsnap_table_hits_f64(
        nat.ptr(table, torch.float64, "table"), nat.ptr(row_offsets, torch.int32, "row_offsets"), B,
        nat.ptr(cuboid, torch.float64, "cuboid"), stride, nat.ptr(hit_mask, torch.int64, "hit_mask"), nat.stream_ptr(table.device))
    return hit_mask


def fixed_pitch(paths, max_wp: int, device) -> tuple[torch.Tensor, torch.Tensor]:
    """Waypoint sets of different lengths -> ([B, max_wp, 3] f64, n_waypoints [B] i32), the in/out layout of minsnap_correct.
    ``paths``: a [B, n, 3] tensor or a sequence of (n_b, 3) arrays / tensors (CUDA tensors are copied on the device)."""
    if isinstance(paths, torch.Tensor) and paths.dim() == 3:
        B, n = paths.shape[0], paths.shape[1]
        wp = torch.zeros((B, max_wp, 3), dtype=torch.float64, device=device)
        wp[:, :n] = paths.to(device=device, dtype=torch.float64)
        return wp, torch.full((B,), n, dtype=torch.int32, device=device)
    counts = [int(len(pth)) for pth in paths]
    if all(isinstance(pth, torch.Tensor) and pth.is_cuda for pth in paths):
        wp = torch.zeros((len(paths), max_wp, 3), dtype=torch.float64, device=device)
        for b, pth in enumerate(paths):
            wp[b, :counts[b]] = pth
        return wp, torch.tensor(counts, dtype=torch.int32, device=device)
    import numpy as np
    host = np.zeros((len(paths), max_wp, 3))
    for b, pth in enumerate(paths):
        host[b, :counts[b]] = pth.detach().cpu().numpy() if isinstance(pth, torch.Tensor) else np.asarray(pth, dtype=float)
    return torch.tensor(host, dtype=torch.float64, device=device), torch.tensor(counts, dtype=torch.int32, device=device)


def minsnap_correct(waypoints: torch.Tensor, n_waypoints: torch.Tensor, velocity: torch.Tensor, dt: float,
                    obstacles: Optional[torch.Tensor] = None, factor: float = START_END_TIME_FACTOR):
    """The whole obstacle-correction loop of MinimumSnap._generate_collision_free_trajectory (minimum_snap.py:63-95) on the
    device: plan, find the splines with a sampled point inside the current obstacle, insert their midpoints, plan again.

    waypoints [B, max_wp, 3] f64 and n_waypoints [B] i32 are updated IN PLACE (fixed pitch, see ``fixed_pitch``); obstacles
    [n_obs, 6] f64 (shared) or [B, n_obs, 6], None / empty = plain plan.  Returns (coeffs [B, max_wp-1, 8, 3], times
    [B, max_wp-1], status [B] i32, rounds).  Synchronises the current stream (uavb.h)."""
    B, max_wp = waypoints.shape[0], waypoints.shape[1]
    dev = waypoints.device
    coeffs = torch.empty((B, max_wp - 1, 8, 3), dtype=torch.float64, device=dev)
    times = torch.empty((B, max_wp - 1), dtype=torch.float64, device=dev)
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    n_obs, stride, obs = 0, 0, None
    if obstacles is not None and obstacles.numel() > 0:
        obs = obstacles.to(device=dev, dtype=torch.float64).contiguous()
        if obs.dim() == 3:
            if obs.shape[0] != B:
                raise ValueError("per-mission obstacles must have shape (B, n_obs, 6)")
            n_obs, stride = int(obs.shape[1]), int(obs.shape[1]) * 6
        else:
            obs = obs.reshape(-1, 6)
            n_obs = int(obs.shape[0])
    rounds = ctypes.c_int(0)
    nat.on(dev).uavb_minsnap_correct_f64(
        nat.ptr(waypoints, torch.float64, "waypoints"), nat.ptr(n_waypoints, torch.int32, "n_waypoints"), nat.ptr(velocity, torch.float64, "velocity"),
        B, max_wp, float(factor), float(dt), nat.ptr(obs), n_obs, stride, nat.ptr(coeffs), nat.ptr(times), nat.ptr(status), ctypes.byref(rounds),
        nat.stream_ptr(dev))
    return coeffs, times, status, rounds.value


def pack_segments(coeffs: torch.Tensor, times: torch.Tensor, n_waypoints: torch.Tensor, n_seg: Optional[int] = None):
    """Fixed pitch -> packed: (coeffs [n_seg, 8, 3], times [n_seg], seg_offsets [B+1] i32) in mission order.
    ``n_seg``: the total spline count when the caller knows it (saves the device->host read)."""
    B, max_wp = coeffs.shape[0], coeffs.shape[1] + 1
    dev = coeffs.device
    seg_offsets = torch.zeros((B + 1,), dtype=torch.int32, device=dev)
    seg_offsets[1:] = torch.cumsum(n_waypoints - 1, 0)
    if n_seg is None:
        n_seg = int(seg_offsets[-1].item())
    c = torch.empty((n_seg, 8, 3), dtype=torch.float64, device=dev)
    t = torch.empty((n_seg,), dtype=torch.float64, device=dev)
    nat.on(dev).uavb_minsnap_pack_f64(nat.ptr(coeffs, torch.float64, "coeffs"), nat.ptr(times, torch.float64, "times"),
                                              nat.ptr(n_waypoints, torch.int32, "n_waypoints"), B, max_wp, nat.ptr(seg_offsets), nat.ptr(c), nat.ptr(t),
                                              nat.stream_ptr(dev))
    return c, t, seg_offsets


class TooManySplines(RuntimeError):
    """The correction loop needed more than UAVB_MAX_SPLINES splines (an obstacle probably contains a waypoint: the reference
    loops forever in that case, minimum_snap.py:80-93)."""


def plan_collision_free(paths, velocity: torch.Tensor, dt: float, obstacles: Optional[torch.Tensor], factor: float = START_END_TIME_FACTOR,
                        device=None):
    """Plan B missions with the reference's correction loop and return them packed:
    (coeffs [n_seg, 8, 3], times [n_seg], seg_offsets [B+1], status [B], waypoints [B, max_wp, 3], n_waypoints [B], rounds).
    The waypoint capacity starts a few midpoints above the longest mission and is raised to the solver's limit once if some
    mission outgrows it; a mission that outgrows UAVB_MAX_SPLINES raises TooManySplines."""
    dev = _dev(device) if not isinstance(paths, torch.Tensor) else paths.device
    longest = int(paths.shape[1]) if isinstance(paths, torch.Tensor) else max(len(p) for p in paths)
    n_seg0 = int(paths.shape[0] * (paths.shape[1] - 1)) if isinstance(paths, torch.Tensor) else sum(len(p) - 1 for p in paths)
    if longest - 1 > nat.MAX_SPLINES:
        raise TooManySplines(f"too many splines ({longest - 1}; the solver accepts at most {nat.MAX_SPLINES})")
    cap = min(nat.MAX_SPLINES + 1, longest + 8)
    while True:
        wp, n_wp = fixed_pitch(paths, cap, dev)
        coeffs, times, status, rounds = minsnap_correct(wp, n_wp, velocity, dt, obstacles, factor)
        if not bool((status == nat.SOLVE_TOO_MANY).any()):
            break
        if cap == nat.MAX_SPLINES + 1:
            bad = int((status == nat.SOLVE_TOO_MANY).nonzero()[0])
            raise TooManySplines(f"mission {bad}: obstacle correction needs more than {nat.MAX_SPLINES} splines -- an obstacle probably "
                                 "contains a waypoint (the reference loops forever in this case)")
        cap = nat.MAX_SPLINES + 1
    c, t, seg_offsets = pack_segments(coeffs, times, n_wp, n_seg0 if rounds <= 1 else None)      # one round: nothing was inserted
    return c, t, seg_offsets, status, wp, n_wp, rounds


# ------------------------------------------------------------------------------------------ missions
@dataclass
class MissionPlan:
    """Packed mission segments in the layout K2 reads (struct uavb_rollout_args, include/uavb.h)."""
    seg_coeffs: torch.Tensor           # [n_seg, 8, 3] f64, MinimumSnap.coeffs rows per spline
    seg_rows: torch.Tensor             # [n_seg] i32
    seg_table: torch.Tensor            # [n_seg] i32, 1 where a MinimumSnap table starts
    seg_yaw0: torch.Tensor             # [n_seg] f64
    dt: float                          # table sampling period (quad.dt * frequency, main.py:97)
    n_seg_shared: int = 0              # > 0: every rollout flies segments [0, n_seg_shared)
    seg_begin: Optional[torch.Tensor] = None   # [B] i32 per-rollout missions
    seg_count: Optional[torch.Tensor] = None   # [B] i32
    rows_per_mission: Optional[torch.Tensor] = None   # [n_missions] i32 table rows of each mission (computed on first use when None)
    times: Optional[torch.Tensor] = None       # [n_seg] f64 (MinimumSnap.times)
    targets: Optional[torch.Tensor] = None     # shared missions: [n_rows, 56] u8 per-row set-points (uavb_rollout_targets_f64)
    status: Optional[torch.Tensor] = None      # shared missions: [n_tables] i32 UAVB_SOLVE_* of each table
    correction_rounds: int = 0                 # plan rounds of the obstacle-correction loop (1 = nothing was hit; 0 = not run)
    report: Optional[torch.Tensor] = None      # speculative shared plan: the pinned control block the correction loop reports into
    report_tables: int = 0
    report_event: Optional[object] = None
    report_ticket: Optional[tuple] = None

    def verify(self) -> None:
        """Speculative shared plans (plan_missions(..., shared=True, obstacles=..., table_rows=...)): wait for the loop's report and
        raise if the plan that was flown is not the one the reference would have produced.  A no-op for every other plan."""
        if self.report is None:
            return
        dev, ticket = self.report_ticket
        if _REPORTS[dev][1] - ticket > _REPORT_RING:
            raise RuntimeError(f"speculative plan: its report block has been handed out again ({_REPORT_RING} plans later); call verify() sooner")
        self.report_event.synchronize()
        r, T = self.report.tolist(), self.report_tables
        if any(r[4:8]):
            raise RuntimeError("speculative plan: the obstacle-correction loop found a sampled point inside a box; plan again without table_rows")
        status, rows = r[8 + T:8 + 2 * T], r[8 + 2 * T:8 + 3 * T]
        if any(status):
            raise RuntimeError(f"speculative plan: solver status {status}")
        if sum(rows) != int(self.rows_per_mission.sum()):
            raise RuntimeError(f"speculative plan: the mission has {sum(rows)} table rows, table_rows said {int(self.rows_per_mission.sum())}")
        self.status = torch.tensor(status, dtype=torch.int32)
        self.report = None

    @property
    def shared(self) -> bool:
        return self.seg_begin is None

    @property
    def total_rows(self) -> torch.Tensor:
        """[n_missions] i32 table rows of each mission."""
        if self.rows_per_mission is None:
            n = 1 if self.shared else self.seg_begin.numel()
            self.rows_per_mission = self.seg_rows.reshape(n, -1).sum(dim=1).to(torch.int32)
        return self.rows_per_mission


def plan_missions(tables: Sequence[tuple[torch.Tensor, torch.Tensor]], dt: float, shared: bool = False,
                  factor: float = START_END_TIME_FACTOR, table_rows: Optional[int] = None, obstacles: Optional[torch.Tensor] = None) -> MissionPlan:
    """Solve and pack missions made of consecutive MinimumSnap tables.

    ``obstacles`` ([n_obs, 6] f64, or [B, n_obs, 6] per mission): every table is planned with the reference's obstacle-correction
    loop (MinimumSnap(path, obstacles, ...).get_trajectory(), minimum_snap.py:63-95, as _generate_mission_trajectory does for
    both tables, main.py:80-83) -- midpoints are inserted where a sampled point lies inside a box, so missions may end up with
    different spline counts.  None plans the given waypoints as they are.

    ``tables`` lists (waypoints [B, S_k+1, 3], velocity [B]) per table, e.g. the vertical take-off
    (S=1) followed by the course of ``_generate_mission_trajectory`` (uav_ac/main.py:73-84).  Mission b
    flies table 0 then table 1 ...; each table keeps its own yaw hold like the reference, where the
    two MinimumSnap instances are independent.  ``shared=True`` requires B == 1 and lets every
    rollout fly the same mission (BASELINE configs[2]); its per-row set-point table is built as well.
    ``table_rows`` (shared only): number of rows to tabulate when the caller already knows the table
    length -- it avoids the device->host read of the row count (rows past the end repeat the last row).
    """
    B = tables[0][0].shape[0]
    dev = tables[0][0].device
    if shared:
        if B != 1:
            raise ValueError("shared=True needs a single mission")
        return _plan_shared(tables, dt, factor, table_rows, obstacles)
    if obstacles is not None and obstacles.numel() > 0:
        return _plan_corrected(tables, dt, factor, obstacles)
    per_table = []
    for wp, vel in tables:
        if wp.shape[0] != B:
            raise ValueError("all tables must have the same batch size")
        S = wp.shape[1] - 1
        coeffs, times, _ = minsnap_solve(wp, vel, factor)
        offs = torch.arange(B + 1, dtype=torch.int32, device=dev) * S
        rows, yaw0, total = table_meta(coeffs, times.reshape(-1), offs, dt)
        flag = torch.zeros((B, S), dtype=torch.int32, device=dev)
        flag[:, 0] = 1
        y0 = torch.zeros((B, S), dtype=torch.float64, device=dev)
        y0[:, 0] = yaw0
        per_table.append((coeffs.reshape(B, S, 8, 3), rows.reshape(B, S), flag, y0, total, times))
    seg_coeffs = torch.cat([t[0] for t in per_table], dim=1).contiguous()
    seg_rows = torch.cat([t[1] for t in per_table], dim=1).contiguous()
    seg_table = torch.cat([t[2] for t in per_table], dim=1).contiguous()
    seg_yaw0 = torch.cat([t[3] for t in per_table], dim=1).contiguous()
    times = torch.cat([t[5] for t in per_table], dim=1).contiguous()
    total = sum(t[4] for t in per_table)
    n_per = seg_rows.shape[1]
    plan = MissionPlan(seg_coeffs.reshape(-1, 8, 3), seg_rows.reshape(-1), seg_table.reshape(-1), seg_yaw0.reshape(-1), float(dt),
                       rows_per_mission=total.to(torch.int32), times=times.reshape(-1))
    plan.seg_begin = torch.arange(B, dtype=torch.int32, device=dev) * n_per
    plan.seg_count = torch.full((B,), n_per, dtype=torch.int32, device=dev)
    return plan


_SHARED_CONSTS: dict = {}


def _plan_corrected(tables, dt: float, factor: float, obstacles: torch.Tensor) -> MissionPlan:
    """Per-rollout missions planned with the correction loop: every table goes through minsnap_correct (ragged spline counts
    afterwards), then the tables of a mission are laid out one after the other in the packed segment arrays."""
    B = tables[0][0].shape[0]
    dev = tables[0][0].device
    per_table = []
    for wp, vel in tables:
        if wp.shape[0] != B:
            raise ValueError("all tables must have the same batch size")
        c, t, seg_off, status, _, n_wp, _ = plan_collision_free(wp, vel, dt, obstacles, factor)
        rows, yaw0, total = table_meta(c, t, seg_off, dt)
        per_table.append((c, t, seg_off.long(), (n_wp - 1).long(), rows, yaw0, total))
    count = sum(p[3] for p in per_table)                                   # segments per mission
    begin = torch.cumsum(count, 0) - count
    n_seg = int(count.sum().item())
    seg_coeffs = torch.empty((n_seg, 8, 3), dtype=torch.float64, device=dev)
    times = torch.empty((n_seg,), dtype=torch.float64, device=dev)
    seg_rows = torch.empty((n_seg,), dtype=torch.int32, device=dev)
    seg_table = torch.zeros((n_seg,), dtype=torch.int32, device=dev)
    seg_yaw0 = torch.zeros((n_seg,), dtype=torch.float64, device=dev)
    within = torch.zeros_like(count)
    arange_b = torch.arange(B, device=dev)
    for c, t, seg_off, S, rows, yaw0, total in per_table:
        owner = torch.repeat_interleave(arange_b, S)                        # mission of every packed segment of this table
        dest = (begin + within)[owner] + (torch.arange(c.shape[0], device=dev) - seg_off[:-1][owner])
        seg_coeffs[dest], times[dest], seg_rows[dest] = c, t, rows
        first = begin + within
        seg_table[first] = 1
        seg_yaw0[first] = yaw0
        within = within + S
    plan = MissionPlan(seg_coeffs, seg_rows, seg_table, seg_yaw0, float(dt), rows_per_mission=sum(p[6] for p in per_table).to(torch.int32), times=times)
    plan.seg_begin = begin.to(torch.int32).contiguous()
    plan.seg_count = count.to(torch.int32).contiguous()
    return plan


_REPORTS: dict = {}


_REPORT_RING = 1024


def _report_block(dev):
    """One [PLAN_REPORT_INTS] row of a pinned ring (_REPORT_RING rows per device) for a speculative plan's report, and its ticket
    (the row is handed out again _REPORT_RING plans later: verify() refuses a plan whose row has been reused)."""
    ring = _REPORTS.get(dev)
    if ring is None:
        ring = _REPORTS[dev] = [torch.zeros((_REPORT_RING, nat.PLAN_REPORT_INTS), dtype=torch.int32).pin_memory(), 0]
    ticket = ring[1]
    ring[1] += 1
    return ring[0][ticket % _REPORT_RING], (dev, ticket)


def _plan_shared_corrected(tables, dt: float, factor: float, table_rows: Optional[int], obstacles: torch.Tensor) -> MissionPlan:
    """uavb_plan_shared_f64: the tables of one mission through the correction loop into the packed segment arrays, one C call
    (a handful of launches, one synchronisation when nothing is hit), then the set-point table.

    With ``table_rows`` (the caller has planned this mission before and knows its table length) the plan is SPECULATIVE: nothing is
    waited for, the kernels of the uncorrected plan are enqueued and the loop's report arrives in pinned memory behind them.
    ``plan.verify()`` -- after the results of the flight have been synchronised -- raises if the correction loop would have inserted
    a midpoint or the table length differs; a Monte-Carlo job that plans the same mission for every batch pays no host round trip."""
    dev = tables[0][0].device
    T = len(tables)
    for wp, vel in tables:
        if wp.shape[0] != 1 or vel.shape != (1,):
            raise ValueError("shared=True needs a single mission per table")
    cap = T * nat.MAX_SPLINES
    coeffs = torch.empty((cap, 8, 3), dtype=torch.float64, device=dev)
    times = torch.empty((cap,), dtype=torch.float64, device=dev)
    rows = torch.empty((cap,), dtype=torch.int32, device=dev)
    seg_table = torch.empty((cap,), dtype=torch.int32, device=dev)
    seg_yaw0 = torch.empty((cap,), dtype=torch.float64, device=dev)
    obs = obstacles.to(device=dev, dtype=torch.float64).contiguous()
    ptrs = (ctypes.c_void_p * T)(*[nat.ptr(wp, torch.float64, "waypoints").value for wp, _ in tables])
    n_wp = (ctypes.c_int * T)(*[int(wp.shape[1]) for wp, _ in tables])
    vels = torch.cat([vel for _, vel in tables]).contiguous() if T > 1 else tables[0][1]
    n_seg, rounds = ctypes.c_int(0), ctypes.c_int(0)
    tab_rows, status = (ctypes.c_int * T)(), (ctypes.c_int * T)()
    report, ticket = _report_block(dev) if table_rows is not None else (None, None)
    nat.on(dev).uavb_plan_shared_f64(T, ptrs, n_wp, nat.ptr(vels, torch.float64, "velocity"), float(factor), float(dt), nat.ptr(obs),
                                     int(obs.shape[0]), cap, nat.ptr(coeffs), nat.ptr(times), nat.ptr(rows), nat.ptr(seg_table),
                                     nat.ptr(seg_yaw0), ctypes.byref(n_seg), tab_rows, status, ctypes.byref(rounds),
                                     ctypes.c_void_p(report.data_ptr()) if report is not None else None, nat.stream_ptr(dev))
    n = n_seg.value
    plan = MissionPlan(coeffs[:n], rows[:n], seg_table[:n], seg_yaw0[:n], float(dt), times=times[:n], n_seg_shared=n)
    if report is not None:
        total = int(table_rows)
        plan.report, plan.report_tables, plan.report_ticket = report, T, ticket
        plan.report_event = torch.cuda.Event()
        plan.report_event.record(torch.cuda.current_stream(dev))
        plan.correction_rounds = 1
    else:
        if any(st == nat.SOLVE_TOO_MANY for st in status):
            raise TooManySplines(f"obstacle correction needs more than {nat.MAX_SPLINES} splines in one table -- an obstacle probably contains a "
                                 "waypoint (the reference loops forever in this case)")
        total = sum(tab_rows)
        plan.status = torch.tensor(list(status), dtype=torch.int32)             # host tensors: the C call already brought them back
        plan.correction_rounds = rounds.value
    plan.rows_per_mission = torch.tensor([total], dtype=torch.int32)
    plan.targets = rollout_targets(plan, total)
    return plan


def _plan_shared(tables, dt: float, factor: float, table_rows: Optional[int], obstacles: Optional[torch.Tensor] = None) -> MissionPlan:
    """One mission flown by every rollout: K1 per table straight into the packed segment arrays, one table-geometry launch,
    the set-point table -- T + 5 kernel launches for T tables, no host synchronisation when ``table_rows`` is given.
    With obstacles the T tables go through the correction loop as a batch of T missions (one extra synchronisation)."""
    dev = tables[0][0].device
    if obstacles is not None and obstacles.numel() > 0:
        if obstacles.dim() != 2:
            raise ValueError("a shared mission takes one obstacle set (n_obs, 6)")
        return _plan_shared_corrected(tables, dt, factor, table_rows, obstacles)
    splines = tuple(int(wp.shape[1]) - 1 for wp, _ in tables)
    n_seg, T = sum(splines), len(splines)
    key = (dev, splines)
    if key not in _SHARED_CONSTS:                       # launch-invariant index arrays, built once per mission shape
        starts = [sum(splines[:k]) for k in range(T)]
        flag = torch.zeros(n_seg, dtype=torch.int32)
        flag[starts] = 1
        _SHARED_CONSTS[key] = (torch.tensor(starts + [n_seg], dtype=torch.int32, device=dev), flag.to(dev), torch.tensor(starts, dtype=torch.int64, device=dev))
    offsets, seg_table, starts = _SHARED_CONSTS[key]
    coeffs = torch.empty((n_seg, 8, 3), dtype=torch.float64, device=dev)
    times = torch.empty((n_seg,), dtype=torch.float64, device=dev)
    status = torch.empty((T,), dtype=torch.int32, device=dev)
    st, off = nat.stream_ptr(dev), 0
    for k, (wp, vel) in enumerate(tables):
        if wp.shape[0] != 1 or vel.shape != (1,):
            raise ValueError("shared=True needs a single mission per table")
        nat.on(dev).uavb_minsnap_solve_f64(nat.ptr(wp, torch.float64, "waypoints"), nat.ptr(vel, torch.float64, "velocity"), 1, splines[k], float(factor),
                                           ctypes.c_void_p(coeffs.data_ptr() + off * 192), ctypes.c_void_p(times.data_ptr() + off * 8),
                                           ctypes.c_void_p(status.data_ptr() + k * 4), st)
        off += splines[k]
    rows, yaw0, total = table_meta(coeffs, times, offsets, dt)
    seg_yaw0 = torch.zeros((n_seg,), dtype=torch.float64, device=dev).index_copy_(0, starts, yaw0)
    plan = MissionPlan(coeffs, rows, seg_table, seg_yaw0, float(dt), times=times, n_seg_shared=n_seg)
    plan.status = status
    plan.targets = rollout_targets(plan, table_rows)
    return plan


def rollout_targets(plan: MissionPlan, n_rows: Optional[int] = None) -> torch.Tensor:
    """Per-row set-points of a shared mission ([n_rows, 56] bytes; struct TargetRow): what every drone of a shared-mission
    rollout reads once per outer period instead of evaluating the polynomials itself (bit-identical results).
    ``n_rows`` defaults to sum(seg_rows), which costs one device->host read."""
    n_seg = plan.seg_rows.numel()
    if n_rows is None:
        n_rows = int(plan.total_rows.sum().item())
    out = torch.empty((n_rows, nat.TARGET_ROW_BYTES), dtype=torch.uint8, device=plan.seg_coeffs.device)
    nat.on(out.device).uavb_rollout_targets_f64(
        nat.ptr(plan.seg_coeffs, torch.float64, "seg_coeffs"), nat.ptr(plan.seg_rows, torch.int32, "seg_rows"), nat.ptr(plan.seg_table, torch.int32, "seg_table"),
        nat.ptr(plan.seg_yaw0, torch.float64, "seg_yaw0"), n_seg, float(plan.dt), nat.ptr(out), n_rows, nat.stream_ptr(out.device))
    return out


# ------------------------------------------------------------------------------------------ caller tables
@dataclass
class TablePlan:
    """Caller-supplied (N, 11) trajectory tables in the layout K2 reads (struct uavb_table_set, include/uavb.h): what
    TrajectoryController(controller, quad, trajectory, frequency) flies (main.py:10-61), for every rollout of a batch."""
    rows: torch.Tensor                           # [n_rows, 56] u8 set-point records (uavb_table_targets_f64), tables one after the other
    rows_per_table: tuple                        # host: rows of every table (known from the input shapes)
    last_position: torch.Tensor                  # [n_tables, 3] f64 position of every table's last row (the default goal)
    offsets: Optional[torch.Tensor] = None       # [n_tables + 1] i64 first row of every table; None = ONE table flown by every rollout
    table_index: Optional[torch.Tensor] = None   # [B] i32 table of every rollout; None = rollout b flies table b

    @property
    def shared(self) -> bool:
        return self.offsets is None

    @property
    def n_tables(self) -> int:
        return len(self.rows_per_table)

    @property
    def max_rows(self) -> int:
        return max(self.rows_per_table)

    def goals(self, B: int) -> torch.Tensor:
        """The last row's position of every rollout's table: [3] for a shared table, else [B, 3]."""
        if self.shared:
            return self.last_position[0].contiguous()
        if self.table_index is None:
            if self.n_tables != B:
                raise ValueError(f"{self.n_tables} tables without table_index need B = {self.n_tables}, got {B}")
            return self.last_position
        return self.last_position.index_select(0, self.table_index.long()).contiguous()


def table_targets(tables: torch.Tensor) -> torch.Tensor:
    """[n_rows, 11] f64 (tables packed one after the other) -> [n_rows, 56] u8 set-point records (uavb_table_targets_f64): x y z
    as given, v / a rounded to fp32, the yaw column as its heading direction (cos, sin)."""
    if tables.dim() != 2 or tables.shape[1] != 11:
        raise ValueError(f"tables must have shape (n_rows, 11), got {tuple(tables.shape)}")
    out = torch.empty((tables.shape[0], nat.TARGET_ROW_BYTES), dtype=torch.uint8, device=tables.device)
    nat.on(tables.device).uavb_table_targets_f64(nat.ptr(tables, torch.float64, "tables"), int(tables.shape[0]), nat.ptr(out),
                                                 nat.stream_ptr(tables.device))
    return out


def plan_tables(tables, table_index=None, device=None) -> TablePlan:
    """Trajectory tables [x y z vx vy vz ax ay az yaw spline_id] for ``rollout``.

    ``tables``: one (N, 11) table, a (T, N, 11) stack, or a sequence of (N_t, 11) tables of different lengths (arrays or tensors).
    One (N, 11) table without ``table_index`` is flown by every rollout (the shared-table kernel); otherwise rollout b flies table
    ``table_index[b]`` ([B] ints in [0, T)), or table b when ``table_index`` is None (then B = T).  Every table needs >= 1 row.
    The yaw column is the set-point itself, as TrajectoryController uses it; spline_id is ignored."""
    import numpy as np

    def as_f64(t):
        return t.detach().to(dtype=torch.float64) if isinstance(t, torch.Tensor) else torch.as_tensor(np.asarray(t, dtype=np.float64))

    single, stack = False, None
    if isinstance(tables, (torch.Tensor, np.ndarray)):
        stack = as_f64(tables)
        if stack.dim() == 2:
            parts, single = [stack], True
        elif stack.dim() == 3:
            parts = list(stack.unbind(0))
        else:
            raise ValueError(f"tables must be (N, 11), (T, N, 11) or a sequence of (N_t, 11) tables, got shape {tuple(stack.shape)}")
    else:
        parts = [as_f64(t) for t in tables]
    if not parts:
        raise ValueError("no tables given")
    for k, t in enumerate(parts):
        if t.dim() != 2 or t.shape[1] != 11:
            raise ValueError(f"table {k} must have shape (N, 11), got {tuple(t.shape)}")
        if t.shape[0] < 1:
            raise ValueError(f"table {k} has no rows")
    if table_index is not None:
        idx = table_index if isinstance(table_index, torch.Tensor) else torch.as_tensor(np.asarray(table_index))
        if idx.dim() != 1 or idx.dtype.is_floating_point or idx.dtype == torch.bool:
            raise ValueError("table_index must be a 1-D integer array of shape (B,)")
        _check_index_range(idx, len(parts))
    dev =torch.device(device) if device is not None else (parts[0].device if parts[0].is_cuda else _dev())
    counts = tuple(int(t.shape[0]) for t in parts)
    if len(parts) == 1:
        packed = parts[0].to(dev).contiguous()
    elif stack is not None:                                                    # a (T, N, 11) stack is already packed
        packed = stack.to(dev).reshape(-1, 11).contiguous()
    else:
        packed = torch.cat([p.to(dev) for p in parts]).contiguous()
    ends = torch.tensor(np.cumsum(counts) - 1, dtype=torch.int64, device=dev)
    plan = TablePlan(table_targets(packed), counts, packed.index_select(0, ends)[:, :3].contiguous())
    if single and table_index is None:
        return plan
    plan.offsets = torch.tensor(np.concatenate(([0], np.cumsum(counts))), dtype=torch.int64, device=dev)
    if table_index is not None:
        plan.table_index = idx.to(device=dev, dtype=torch.int32).contiguous()
    return plan


def _check_index_range(idx: torch.Tensor, n_tables: int) -> None:
    """0 <= idx < n_tables: one reduction (on the device for a CUDA tensor, one read back)."""
    if idx.numel() == 0:
        return
    lo, hi = torch.stack(torch.aminmax(idx)).tolist()
    if lo < 0 or hi >= n_tables:
        raise ValueError(f"table_index must lie in [0, {n_tables}), got values in [{lo}, {hi}]")


# ------------------------------------------------------------------------------------------ K2
@dataclass
class RolloutResult:
    metrics: Optional[torch.Tensor]    # [B, 8]: final_dist, collision, rmse, mean_err, max_err, status, first_hit, periods
    state: Optional[torch.Tensor]      # [13, B] final X (SoA)
    log: Optional[torch.Tensor]        # [n_samples, 13, B]
    carry: Optional[torch.Tensor]      # [48, B] resumable block
    n_ticks: int = 0
    traj: Optional[torch.Tensor] = None        # [traj_max_samples, 3, B] gated 20 Hz positions (mujoco_sim.py:201-218)
    traj_count: Optional[torch.Tensor] = None  # [B] i32 samples the reference would hold


def rollout(plan, B: int, n_ticks: int, *, start: torch.Tensor, goal: Optional[torch.Tensor] = None,
            vehicle: Optional[nat.Vehicle] = None, frequency: int = 10, mc_mass: Optional[torch.Tensor] = None,
            mc_inertia: Optional[torch.Tensor] = None, mc_gains: Optional[torch.Tensor] = None, mc_wind: Optional[torch.Tensor] = None,
            obstacles: Optional[torch.Tensor] = None, obstacle_set: Optional[torch.Tensor] = None, thrust_frame_lag: int = 1,
            log_stride: int = 0, carry: Optional[torch.Tensor] = None, resume: bool = False, want_state: bool = True,
            want_metrics: bool = True, want_carry: bool = False, dtype: torch.dtype = torch.float32, index_base: int = 0, use_targets: bool = True,
            out: Optional[RolloutResult] = None, n_slices: int = 0, log_tma: int = 0, ground_z: Optional[float] = None,
            traj_max_samples: int = 0, traj_gate_z: float = 0.0, traj_interval: float = 0.05, pair_kernel_only: bool = False) -> RolloutResult:
    """n_ticks ticks of `trajectory_controller.step(); simulation.step()` for B drones
    (tests/integration/test_mujoco_trajectory_tracking.py:27-31) in one persistent kernel launch.

    start / goal: [3] or [B, 3] f64.  mc_mass [B], mc_inertia [3, B], mc_gains [11, B], mc_wind [3, B] f32 (SoA).
    obstacles: [n_obs, 6] (shared) or [n_sets, n_obs, 6] f32 with obstacle_set [B] i32.
    dtype float64 selects the validation kernel (outputs f64, no carry).
    n_slices > 0 forces the number of time slices of the fp32 launch (uavb.h; results do not depend on it).
    log_tma = -1 writes the state log with per-thread stores instead of staged TMA tensor stores (uavb.h; same bits).
    ground_z: optional unilateral floor (NED; uavb.h ground_on / ground_z).  traj_max_samples > 0 also records the viewer's
    flown-path list (MujocoSimulation._record_actual_trajectory, mujoco_sim.py:201-218): positions every traj_interval seconds
    of simulation time while z <= traj_gate_z, into result.traj [traj_max_samples, 3, B] / result.traj_count [B].
    ``plan``: a MissionPlan (waypoint missions), or a TablePlan (``plan_tables``: caller trajectory tables, one row per
    ``frequency`` ticks; fp32 only).  A MissionPlan's table period ``plan.dt`` must equal ``vehicle.dt * frequency`` (to 1e-12
    relative): it is also the outer-loop dt of the controller (altitude integral, set-point times), which the reference takes as
    ``quad.dt * frequency`` for both (main.py:97); a mismatch raises ValueError.  A TablePlan takes its outer dt from
    ``vehicle.dt * frequency``.
    """
    tables = isinstance(plan, TablePlan)
    dev = plan.rows.device if tables else plan.seg_coeffs.device
    f64 = dtype == torch.float64
    if tables and f64:
        raise ValueError("trajectory tables fly in the fp32 rollout only (uavb_rollout_f64 takes waypoint missions)")
    veh = vehicle if vehicle is not None else nat.default_vehicle()
    if not tables and frequency >= 1 and abs(plan.dt - veh.dt * frequency) > 1e-12 * abs(veh.dt * frequency):
        raise ValueError(f"the plan is sampled at dt = {plan.dt}, but vehicle.dt * frequency = {veh.dt} * {frequency} = {veh.dt * frequency}: "
                         "plan the mission at vehicle.dt * frequency")
    odt = torch.float64 if f64 else torch.float32
    a = nat.RolloutArgs()
    a.B, a.n_ticks, a.inner_per_outer = int(B), int(n_ticks), int(frequency)
    a.thrust_frame_lag, a.resume, a.log_stride = int(thrust_frame_lag), int(bool(resume)), int(log_stride)
    a.index_base = int(index_base)
    a.n_slices = int(n_slices)
    a.log_tma = int(log_tma)
    a.pair_kernel_only = int(bool(pair_kernel_only))
    if ground_z is not None:
        a.ground_on, a.ground_z = 1, float(ground_z)
    a.veh = veh
    a.mc_mass = nat.ptr(mc_mass, torch.float32, "mc_mass")
    a.mc_inertia = nat.ptr(mc_inertia, torch.float32, "mc_inertia")
    a.mc_gains = nat.ptr(mc_gains, torch.float32, "mc_gains")
    a.mc_wind = nat.ptr(mc_wind, torch.float32, "mc_wind")
    for name, t, shape in (("mc_mass", mc_mass, (B,)), ("mc_inertia", mc_inertia, (3, B)), ("mc_gains", mc_gains, (nat.N_GAINS, B)),
                           ("mc_wind", mc_wind, (3, B))):
        if t is not None and tuple(t.shape) != shape:
            raise ValueError(f"{name} must have shape {shape}, got {tuple(t.shape)}")
    ts = nat.TableSet()
    if tables:                                        # every mission-segment field stays NULL / 0 (uavb_rollout_tables_f32)
        ts.rows = nat.ptr(plan.rows, torch.uint8, "rows")
        if plan.shared:
            ts.shared_rows = int(plan.rows.shape[0])
        else:
            ts.offsets = nat.ptr(plan.offsets, torch.int64, "offsets")
            ts.n_tables = plan.n_tables
            if plan.table_index is not None:
                if plan.table_index.numel() != B:
                    raise ValueError(f"table_index holds {plan.table_index.numel()} rollouts, B = {B}")
                ts.table_index = nat.ptr(plan.table_index, torch.int32, "table_index")
            elif plan.n_tables != B:
                raise ValueError(f"{plan.n_tables} tables without table_index need B = {plan.n_tables}, got {B}")
    else:
        a.seg_coeffs = nat.ptr(plan.seg_coeffs, torch.float64, "seg_coeffs")
        a.seg_rows = nat.ptr(plan.seg_rows, torch.int32, "seg_rows")
        a.seg_table = nat.ptr(plan.seg_table, torch.int32, "seg_table")
        a.seg_yaw0 = nat.ptr(plan.seg_yaw0, torch.float64, "seg_yaw0")
        if plan.shared:
            a.n_seg_shared = int(plan.n_seg_shared)
            if plan.targets is not None and use_targets:
                a.shared_targets = nat.ptr(plan.targets, torch.uint8, "targets")
                a.n_target_rows = int(plan.targets.shape[0])
        else:
            if plan.seg_begin.numel() != B:
                raise ValueError("plan holds per-rollout missions for a different batch size")
            a.mission_seg_begin = nat.ptr(plan.seg_begin, torch.int32, "seg_begin")
            a.mission_seg_count = nat.ptr(plan.seg_count, torch.int32, "seg_count")
        a.dt_outer = float(plan.dt)
    a.start = nat.ptr(start, torch.float64, "start")
    a.start_stride = 0 if start.dim() == 1 else 3
    if goal is not None:
        a.goal = nat.ptr(goal, torch.float64, "goal")
        a.goal_stride = 0 if goal.dim() == 1 else 3
    if obstacles is not None and obstacles.numel() > 0:
        obs = obstacles if obstacles.dim() == 3 else obstacles.unsqueeze(0)
        obs = obs.to(torch.float32).contiguous()
        a.n_obs_sets, a.n_obs = int(obs.shape[0]), int(obs.shape[1])
        a.aabbs = nat.ptr(obs, torch.float32, "obstacles")
        if obstacle_set is not None:
            a.aabb_set = nat.ptr(obstacle_set, torch.int32, "obstacle_set")
        elif obs.shape[0] != 1:
            raise ValueError("several obstacle sets need obstacle_set")
    res = out if out is not None else RolloutResult(None, None, None, None)
    res.n_ticks = int(n_ticks)
    if want_metrics and res.metrics is None:
        res.metrics = torch.empty((B, nat.N_METRICS), dtype=odt, device=dev)
    if want_state and res.state is None:
        res.state = torch.empty((nat.STATE_DIM, B), dtype=odt, device=dev)
    if log_stride > 0 and res.log is None:
        res.log = torch.empty((n_ticks // log_stride, nat.STATE_DIM, B), dtype=odt, device=dev)
    if resume:
        if carry is None:
            raise ValueError("resume=True needs the carry block of the previous launch")
        res.carry = carry
    elif (want_carry or carry is not None) and not f64:
        res.carry = carry if carry is not None else torch.empty((nat.CARRY_WORDS, B), dtype=torch.float32, device=dev)
    a.carry = nat.ptr(res.carry, torch.float32, "carry")
    a.state_out = nat.ptr(res.state if want_state else None)
    a.metrics_out = nat.ptr(res.metrics if want_metrics else None)
    a.log_out = nat.ptr(res.log if log_stride > 0 else None)
    if traj_max_samples > 0:
        if res.traj is None:
            res.traj = torch.zeros((int(traj_max_samples), 3, B), dtype=torch.float32, device=dev)
            res.traj_count = torch.zeros((B,), dtype=torch.int32, device=dev)
        a.traj_out, a.traj_count_out = nat.ptr(res.traj, torch.float32, "traj"), nat.ptr(res.traj_count, torch.int32, "traj_count")
        a.traj_max_samples, a.traj_gate_z, a.traj_interval = int(res.traj.shape[0]), float(traj_gate_z), float(traj_interval)
    with torch.cuda.device(dev):                      # the library works on the CURRENT device: make it the tensors' device
        if tables:
            nat.check(nat.lib().uavb_rollout_tables_f32(ctypes.byref(a), ctypes.byref(ts), nat.stream_ptr(dev)), "uavb_rollout_tables_f32")
        else:
            fn = nat.lib().uavb_rollout_f64 if f64 else nat.lib().uavb_rollout_f32
            nat.check(fn(ctypes.byref(a), nat.stream_ptr(dev)), "uavb_rollout_f64" if f64 else "uavb_rollout_f32")
    return res


# ------------------------------------------------------------------------------------------ Monte-Carlo inputs
def mc_uniform(seed: int, B: int, lo: Sequence[float], hi: Sequence[float], *, index_base: int = 0, stream_id: int = 0,
               device=None) -> torch.Tensor:
    """[n_fields, B] f32 with field k uniform in (lo[k], hi[k]); Philox keyed by (seed, global index)."""
    dev = _dev(device)
    lo_t = torch.tensor(list(lo), dtype=torch.float32, device=dev)
    hi_t = torch.tensor(list(hi), dtype=torch.float32, device=dev)
    out = torch.empty((lo_t.numel(), B), dtype=torch.float32, device=dev)
    nat.on(dev).uavb_mc_uniform_f32(int(seed), int(index_base), int(stream_id), int(B), int(lo_t.numel()), nat.ptr(lo_t), nat.ptr(hi_t),
                                            nat.ptr(out), nat.stream_ptr(dev))
    return out


def mc_missions(seed: int, B: int, S: int = 4, *, index_base: int = 0, device=None):
    """BASELINE configs[1] generator on the device: waypoints [B, S+1, 3] f64, velocity [B] f64."""
    dev = _dev(device)
    wp = torch.empty((B, S + 1, 3), dtype=torch.float64, device=dev)
    vel = torch.empty((B,), dtype=torch.float64, device=dev)
    nat.on(dev).uavb_mc_missions_f64(int(seed), int(index_base), int(B), int(S), nat.ptr(wp), nat.ptr(vel), nat.stream_ptr(dev))
    return wp, vel
