// Host build of csrc/rollout_core.cuh (not product, never loaded by the package): the scalar mission loop rollout_run<double> --
// outer/inner schedule, table cursor, metrics, collision flag -- at any outer-loop frequency, so that tests/test_frequency_host.py
// can compare the schedule logic with the fp64 C oracle without a GPU.
//   g++ -O2 -shared -fPIC -std=c++17 -I uav-autonomous-control_b200/csrc tests/devtools/host_rollout.cpp -o /tmp/libhost_rollout.so
#include <cmath>
#include <cstring>
#include "rollout_core.cuh"
#include "veh_setup.cuh"

using namespace uavb;

// Inclusive point-in-AABB boxes and the Chebyshev gap to the nearest one, as BoxesT (rollout_impl.cuh) computes them.
struct HostBoxes {
  static constexpr bool kAny = true;
  const double* b;
  int n;
  bool hit(double x, double y, double z) const {
    for (int i = 0; i < n; ++i) {
      const double* q = b + 6 * i;
      if (q[0] <= x && x <= q[1] && q[2] <= y && y <= q[3] && q[4] <= z && z <= q[5]) return true;
    }
    return false;
  }
  double gap(double x, double y, double z) const {
    double g = 3.0e38;
    for (int i = 0; i < n; ++i) {
      const double* q = b + 6 * i;
      const double gi = fmax(fmax(fmax(q[0] - x, x - q[1]), fmax(q[2] - y, y - q[3])), fmax(q[4] - z, z - q[5]));
      g = (gi < g || gi != gi) ? gi : g;
    }
    return g;
  }
};

// The state after every `stride` ticks; the quaternion is renormalised in every tick, as in the logging kernels.
struct HostLog {
  static constexpr bool kNormEveryTick = true;
  double* out;
  int stride, left;
  void tick(const Drone<double>& d) {
    if (--left) return;
    left = stride;
    const double x[13] = {d.px + d.dx, d.py + d.dy, d.pz + d.dz, d.q0, d.q1, d.q2, d.q3, d.vx, d.vy, d.vz, d.wx, d.wy, d.wz};
    memcpy(out, x, sizeof(x));
    out += 13;
  }
};

// One drone on a packed mission (segments in the layout of uavb_rollout_args), `freq` ticks per outer period, flown as two calls of
// rollout_run split after `split` ticks (0 <= split <= n_ticks; the second call resumes from the first one's drone, cursor and
// accumulators, as a chunked launch does).  mc[18]: mass scale, inertia scale[3], gain scale[11], wind force[3].
// metrics[8] as UAVB_M_*; X[13] the final state; log (log_stride > 0): [n_ticks / log_stride][13].
extern "C" int host_rollout(const double* coeffs, const int* rows, const int* table, const double* yaw0, int n_seg, const double* start, int freq,
                            int n_ticks, int split, int lag, const double* boxes, int n_boxes, const double* goal, const double* mc, double* metrics,
                            double* X, int log_stride, double* log) {
  if (freq < 1 || n_seg < 1 || split < 0 || split > n_ticks) return 1;
  uavb_vehicle uv;
  vehicle_defaults(&uv);
  McValues o;
  o.mass = uv.mass * mc[0];
  for (int i = 0; i < 3; ++i) o.inertia[i] = uv.inertia[i] * mc[1 + i];
  for (int i = 0; i < UAVB_N_GAINS; ++i) o.gains[i] = uv.gains[i] * mc[4 + i];
  for (int i = 0; i < 3; ++i) o.wind[i] = mc[15 + i];
  const double dt_outer = uv.dt * freq;
  VehU<double> u;
  make_vehu<double>(u, uv, dt_outer);
  VehP<double> v;
  make_vehp<double>(v, uv, o);
  MissionView m{};
  m.coeffs = coeffs; m.rows = rows; m.table = table; m.yaw0 = yaw0;
  m.seg_begin = 0; m.seg_count = n_seg; m.dt_outer = dt_outer;
  Drone<double> d;
  Cursor<double> c;
  Accum<double> a;
  drone_init<double>(d, u, start[0], start[1], start[2]);
  cursor_init<double>(c);
  accum_init<double>(a);
  const HostBoxes obst{boxes, n_boxes};
  const bool logging = log_stride > 0;
  HostLog lg{log, log_stride, log_stride};
  NoLog nl;
  for (int part = 0; part < 2; ++part) {
    const int t0 = part ? split : 0, n = part ? n_ticks - split : split;
    if (logging) rollout_run<double>(d, c, a, u, v, m, t0, n, freq, lag, obst, lg);
    else rollout_run<double>(d, c, a, u, v, m, t0, n, freq, lag, obst, nl);
  }
  // write_outputs (rollout_impl.cuh)
  const double fx = d.px + d.dx, fy = d.py + d.dy, fz = d.pz + d.dz;
  if (!logging && c.phase != 0) renormalise_q<double>(d);
  const double x[13] = {fx, fy, fz, d.q0, d.q1, d.q2, d.q3, d.vx, d.vy, d.vz, d.wx, d.wy, d.wz};
  memcpy(X, x, sizeof(x));
  const double np = a.periods > 0 ? 1.0 / a.periods : 0.0;
  metrics[UAVB_M_FINAL_DIST] = sqrt((goal[0] - fx) * (goal[0] - fx) + (goal[1] - fy) * (goal[1] - fy) + (goal[2] - fz) * (goal[2] - fz));
  metrics[UAVB_M_COLLISION] = a.collided;
  metrics[UAVB_M_RMSE] = sqrt(a.sum_e2 * np);
  metrics[UAVB_M_MEAN_ERR] = a.sum_e * np;
  metrics[UAVB_M_MAX_ERR] = a.max_e;
  metrics[UAVB_M_STATUS] = a.status;
  metrics[UAVB_M_FIRST_HIT] = a.first_hit;
  metrics[UAVB_M_PERIODS] = a.periods;
  return 0;
}
