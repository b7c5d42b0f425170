// rollout_core.cuh -- the persistent per-drone mission loop of K2: table cursor, outer/inner
// schedule, tracking metrics, collision flag.  Used by rollout_kernels.cu (one thread per drone).
//
// Schedule reproduced (paths relative to /root/reference):
//   TrajectoryController.step (uav_ac/main.py:37-45): outer loop iff inner_step % frequency == 0,
//   using table row `trajectory_index`, then index = min(index+1, N-1) (:61); body-rate loop and
//   set_propeller_speed every tick; then MujocoSimulation.step (mujoco_sim.py:144-151).
//   Tracking error |p - target[:3]| after each outer period (tests/integration/
//   test_mujoco_trajectory_tracking.py:27-31); final distance to goal (main.py:115).
//   Collision flag: inclusive point-in-AABB of minimum_snap.py:327-357 on the body origin after
//   every tick, sticky (BASELINE.json north_star; replaces MuJoCo contacts, mujoco_sim.py:220-230).
#pragma once

#include "flight_core.cuh"

namespace uavb {

// Packed mission segments, reference coefficient layout (MinimumSnap.coeffs rows 8*i+j, 3 axes).
struct MissionView {
  const double* coeffs;   // [n_seg][24]
  const int* rows;        // [n_seg] rows of each segment = len(np.arange(0, T_i, dt)) (minimum_snap.py:104)
  const int* table;       // [n_seg] 1 = first segment of a MinimumSnap table
  const double* yaw0;     // [n_seg] look-ahead yaw of the table starting here (minimum_snap.py:134-135)
  int seg_begin, seg_count;
  double dt_outer;
  // shared missions: the set-points of every table row precomputed once per launch (same arithmetic as cursor_target, so
  // both forms give bit-identical rollouts); the cursor is then just the global row index.  nullptr = evaluate on the fly.
  const TargetRow* trows;
  int n_trows;
  // on-the-fly evaluation: per-thread staging area for the 24 coefficients of the current spline (element k at
  // cache[k * cache_stride]; shared memory in the rollout kernels), refilled only when the spline changes -- a spline
  // lasts ~100-250 outer periods.  nullptr = read the coefficients from global memory every period.
  double* cache;
  int cache_stride;
};

constexpr double kSpeed2Min = 0x1.0c6f7a0b5ed8dp-20;

UAVB_HD double speed2_unfused(double vx, double vy) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy));
#else
  volatile double a = vx * vx, b = vy * vy;          // keep the two products rounded separately (no FMA contraction)
  return a + b;
#endif
}

template <bool V> struct BoolC {
  static constexpr bool value = V;
};

template <class R> struct Cursor {
  int seg, row;           // table row the NEXT outer update will use (main.py:48 trajectory_index)
  int cached_seg;         // packed segment whose coefficients sit in MissionView::cache (-1 = none; not part of the carry)
  int phase;              // inner_step % frequency (main.py:25,39), kept incrementally
  R hx, hy;               // heading direction of the last valid row (minimum_snap.py:126-136 hold-last-valid),
                          // any positive multiple of (cos yaw, sin yaw)
  R ex, ey, ez;           // position error (set-point - position, formed in fp64 and rounded once) at the start of the current
                          // outer period: what the controller saw; the tracking error at its end is this minus the displacement
};

template <class R> struct Accum {
  R sum_e, sum_e2, max_e;
  int periods;
  int collided, first_hit;
  int status;
};

// Loggers see the state after every tick.  kNormEveryTick: renormalise the quaternion in every tick (what a per-tick log
// must show, mujoco_sim.py:36-42) instead of once per outer period (metrics-only rollouts, see physics_step).
struct NoLog {
  static constexpr bool kNormEveryTick = false;
  template <class R> UAVB_HD void tick(const Drone<R>&) {}
};

// Optional unilateral floor (uavb_rollout_args.ground_on / ground_z): NED, z <= ground z.  The floor takes part in the obstacle
// culling below like one more box -- a drone that cannot reach it during a stretch is not tested against it.
struct Ground {
  int on;
  double z;
};

struct NoObstacles {
  static constexpr bool kAny = false;
  template <class R> UAVB_HD R gap(R, R, R) const { return R(3.0e38); }
  template <class R> UAVB_HD bool hit(R, R, R) const { return false; }
};

// Advance the cursor one row with the end clamp of main.py:61.
UAVB_HD void cursor_advance(int* seg, int* row, const MissionView& m) {
  if (*row + 1 < m.rows[m.seg_begin + *seg]) { ++*row; return; }
  int s = *seg + 1;
  while (s < m.seg_count && m.rows[m.seg_begin + s] <= 0) ++s;   // zero-length segments own no rows
  if (s < m.seg_count) { *seg = s; *row = 0; }
}

// Fetch the set-point of the cursor row: polynomial values plus the yaw rule of _calculate_yaws.
template <class R> UAVB_HD void cursor_target(Cursor<R>& c, const MissionView& m, Target<R>* t) {
  const int sg = m.seg_begin + c.seg;
  const double* cf = m.coeffs + (size_t)sg * 24;
  double p[3], v[3], a[3];
  if (m.cache) {
    if (c.cached_seg != sg) {
#if defined(__CUDA_ARCH__)
#pragma unroll
      for (int k = 0; k < 24; ++k) m.cache[k * m.cache_stride] = __ldg(cf + k);
#else
      for (int k = 0; k < 24; ++k) m.cache[k * m.cache_stride] = cf[k];
#endif
      c.cached_seg = sg;
    }
    const double* cc = m.cache;
    const int cs = m.cache_stride;
    eval_row([cc, cs](int i) { return cc[i * cs]; }, (double)c.row * m.dt_outer, p, v, a);
  } else {
#if defined(__CUDA_ARCH__)
    eval_row([cf](int i) { return __ldg(cf + i); }, (double)c.row * m.dt_outer, p, v, a);
#else
    eval_row([cf](int i) { return cf[i]; }, (double)c.row * m.dt_outer, p, v, a);
#endif
  }
  if (c.row == 0 && m.table[sg]) {                       // a new table starts: rows before its first valid row take yaw0
    double s0, c0;
    const double y0 = m.yaw0[sg];
    s0 = sin(y0); c0 = cos(y0);
    c.hx = (R)c0; c.hy = (R)s0;
  }
  // valid iff np.linalg.norm(v_xy) >= 1e-3 (:128-129): norm = sqrt(fl(fl(vx^2) + fl(vy^2))), and sqrt is monotonic, so the
  // test is s >= kSpeed2Min with kSpeed2Min the smallest double whose square root rounds to >= 1e-3.
  if (speed2_unfused(v[0], v[1]) >= kSpeed2Min) { c.hx = (R)v[0]; c.hy = (R)v[1]; }
  t->x = p[0]; t->y = p[1]; t->z = p[2];
  t->vx = (R)v[0]; t->vy = (R)v[1]; t->vz = (R)v[2];
  t->ax = (R)a[0]; t->ay = (R)a[1]; t->az = (R)a[2];
  t->yc = c.hx; t->ys = c.hy;
}

// The same from a precomputed row (shared missions).
template <class R> UAVB_HD void table_target(const TargetRow* rows, int row, Target<R>* t) {
  const TargetRow* r = rows + row;
#if defined(__CUDA_ARCH__)
  t->x = __ldg(&r->x); t->y = __ldg(&r->y); t->z = __ldg(&r->z);
  t->vx = (R)__ldg(&r->vx); t->vy = (R)__ldg(&r->vy); t->vz = (R)__ldg(&r->vz);
  t->ax = (R)__ldg(&r->ax); t->ay = (R)__ldg(&r->ay); t->az = (R)__ldg(&r->az);
  t->yc = (R)__ldg(&r->yc); t->ys = (R)__ldg(&r->ys);
#else
  t->x = r->x; t->y = r->y; t->z = r->z;
  t->vx = (R)r->vx; t->vy = (R)r->vy; t->vz = (R)r->vz; t->ax = (R)r->ax; t->ay = (R)r->ay; t->az = (R)r->az;
  t->yc = (R)r->yc; t->ys = (R)r->ys;
#endif
}

// n_ticks ticks of the closed loop for one drone.  `tick0` is the global index of the first tick
// (first_hit and the log phase are relative to the start of the mission, not of this launch).
// The tick loop is split at outer-period boundaries so the 1 kHz body stays branch-light.
//
// Obstacle culling: during a stretch of n <= freq ticks the drone can move at most
//     reach = (|v| + acc_max n dt) n dt
// (acc_max bounds gravity + full thrust + wind) in any axis.  `clear` is a lower bound of the Chebyshev gap between the
// body origin and the nearest box: it is measured, then only charged with the reach of every stretch flown, and measured
// again when the next stretch could use it up.  While clear > reach no box can be entered before the next check and the
// per-tick inclusive point-in-AABB test (minimum_snap.py:352-357) is skipped for the stretch.  The flag and first-hit tick
// are those of the per-tick test; only the work changes.
// Set-points are evaluated from the mission's splines (cursor_target).
template <class R, class OBST, class LOG>
UAVB_HD void rollout_run(Drone<R>& d, Cursor<R>& c, Accum<R>& a, const VehU<R>& u, const VehP<R>& v, const MissionView& m,
                         int tick0, int n_ticks, int freq, int lag, const OBST& obst, LOG& logger, const Ground gr = Ground{0, 0.0}) {
  typedef Math<R> M;
  int k = 0;
  R clear = R(0);                                            // not part of the carry: every launch / slice measures first
  while (k < n_ticks) {
    if (c.phase == 0) {
      Target<R> t;
      cursor_target<R>(c, m, &t);
      cursor_advance(&c.seg, &c.row, m);
      c.ex = (R)(t.x - d.px); c.ey = (R)(t.y - d.py); c.ez = (R)(t.z - d.pz);   // the position is folded here (d.dx = 0)
      outer_update<R>(d, u, v, t, c.ex, c.ey, c.ez);
    }
    const int n = (freq - c.phase < n_ticks - k) ? (freq - c.phase) : (n_ticks - k);
    bool watch = false;
    if (OBST::kAny && (!a.collided || gr.on)) {
      const R T = (R)n * u.dt;
      const R speed = M::sqrt_fast(d.vx * d.vx + d.vy * d.vy + d.vz * d.vz);
      const R reach = R(1.01) * (speed + v.acc_max * T) * T + R(1e-4);
      if (!(clear > reach)) {
        clear = a.collided ? R(3.0e38) : obst.gap((R)(d.px + (double)d.dx), (R)(d.py + (double)d.dy), (R)(d.pz + (double)d.dz));
        if (gr.on) {
          const R gg = (R)(gr.z - (d.pz + (double)d.dz));  // room above the floor
          clear = (gg < clear || gg != gg) ? gg : clear;
        }
      }
      watch = !(clear > reach);                              // NaN positions keep measuring and watching
      clear -= reach;
    }
#if defined(__CUDA_ARCH__)
    // one decision per warp: with per-rollout missions / obstacle sets the lanes disagree, and a divergent warp would run the
    // whole 1 kHz stretch twice (once per side).  Watching is always correct (the per-tick test is the exact one), so any lane
    // that needs it switches it on for its warp.
    if (OBST::kAny) watch = __any_sync(__activemask(), watch);
#endif
    // the stretch is specialised on the two warp-uniform switches (watch, lag): the 1 kHz body then carries no selects for them
    auto stretch = [&](auto watch_c, auto lag_c) {
      constexpr bool kWatch = decltype(watch_c)::value, kLag = decltype(lag_c)::value;
#if defined(__CUDA_ARCH__)
#pragma unroll 2
#endif
      for (int j = 0; j < n; ++j) {
        inner_tick<R, LOG::kNormEveryTick>(d, u, v, kLag);
        if constexpr (kWatch) {
          if (gr.on && d.pz + (double)d.dz > gr.z) {         // below the floor: back onto it, no downward velocity
            d.dz = (R)(gr.z - d.pz);
            d.vz = M::fmin(d.vz, R(0));
          }
          if (!a.collided && obst.hit((R)(d.px + (double)d.dx), (R)(d.py + (double)d.dy), (R)(d.pz + (double)d.dz))) {
            a.collided = 1; a.first_hit = tick0 + k + j;
          }
        }
        logger.tick(d);
      }
    };
    if (watch) {
      if (lag) stretch(BoolC<true>{}, BoolC<true>{}); else stretch(BoolC<true>{}, BoolC<false>{});
    } else {
      if (lag) stretch(BoolC<false>{}, BoolC<true>{}); else stretch(BoolC<false>{}, BoolC<false>{});
    }
    k += n;
    c.phase += n;
    if (c.phase == freq) {
      c.phase = 0;
      if (!LOG::kNormEveryTick) renormalise_q<R>(d);         // once per outer period (not per launch: chunked runs stay bit-identical)
      // tracking error |set-point - p| after the period (test_mujoco_trajectory_tracking.py:27-31): p = fold + displacement
      const R ex = c.ex - d.dx, ey = c.ey - d.dy, ez = c.ez - d.dz;
      fold_position<R>(d);
      const R e2 = ex * ex + ey * ey + ez * ez;
      const R e = M::sqrt_fast(e2);
      a.sum_e += e; a.sum_e2 += e2; a.max_e = M::fmax(a.max_e, e);
      ++a.periods;
    }
  }
  // status once per call: a non-finite error makes the sum of squares non-finite for good; max_e ignores NaN but keeps Inf
  if (!M::finite(a.sum_e2)) a.status |= 1;
  if (a.max_e > R(1e4)) a.status |= 2;                       // more than 1e4 m from its set-point
}

template <class R> UAVB_HD void drone_init(Drone<R>& d, const VehU<R>& u, double sx, double sy, double sz) {
  d.px = sx; d.py = sy; d.pz = sz;
  d.dx = d.dy = d.dz = R(0);
  d.q0 = R(1); d.q1 = d.q2 = d.q3 = R(0);            // quad.py:78-80
  d.vx = d.vy = d.vz = R(0);
  d.wx = d.wy = d.wz = R(0);
  d.om0 = d.om1 = d.om2 = d.om3 = R(0);              // quad.py:85
  d.integral = R(0);                                 // controller.py:20
  set_thrust_cmd<R>(d, u, R(0));                     // main.py:26
  d.pc = d.qc = d.rc = R(0);                         // main.py:27
  d.cp = d.cq = d.cr = R(0);
  half_axis<R>(d, &d.zbx, &d.zby, &d.zbz);           // mj_forward in MujocoSimulation.__init__ (mujoco_sim.py:81)
}

template <class R> UAVB_HD void cursor_init(Cursor<R>& c) {
  c.seg = 0; c.row = 0; c.cached_seg = -1; c.phase = 0; c.hx = R(1); c.hy = R(0); c.ex = c.ey = c.ez = R(0);
}

template <class R> UAVB_HD void accum_init(Accum<R>& a) {
  a.sum_e = a.sum_e2 = a.max_e = R(0);
  a.periods = 0; a.collided = 0; a.first_hit = -1; a.status = 0;
}

}  // namespace uavb
