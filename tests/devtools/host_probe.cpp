// host_probe.cpp -- DEVELOPMENT NUMERICS PROBE, not part of the product and never loaded by it.
// Compiles the per-drone arithmetic of csrc/flight_core.cuh / rollout_core.cuh for the HOST with g++
// so the fp32 error budget (DESIGN.md) can be explored in the GPU-less build container before GPU
// time is spent.  Host float arithmetic is not bit-identical to the device (FMA contraction, rsqrt,
// __fdividef differ), so this only bounds the error statistically; the parity tests run on the GPU.
//   g++ -O2 -ffp-contract=fast -march=native -I uav-autonomous-control_b200/csrc tests/devtools/host_probe.cpp -o /tmp/host_probe
//   /tmp/host_probe mission.bin out.bin [f32|f64]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "rollout_core.cuh"
#include "veh_setup.cuh"
#include "../../include/uavb.h"

using namespace uavb;

template <class R> struct VecLog {
  static constexpr bool kNormEveryTick = false;
  std::vector<double>* out; int stride; int left;
  void tick(const Drone<R>& d) {
    if (--left) return;
    left = stride;
    double x[17] = {d.px + (double)d.dx, d.py + (double)d.dy, d.pz + (double)d.dz,
                    (double)d.q0, (double)d.q1, (double)d.q2, (double)d.q3, (double)d.vx, (double)d.vy, (double)d.vz,
                    (double)d.wx, (double)d.wy, (double)d.wz, (double)d.om0, (double)d.om1, (double)d.om2, (double)d.om3};
    out->insert(out->end(), x, x + 17);
  }
};

template <class R> int run(const char* in, const char* outp) {
  FILE* f = fopen(in, "rb");
  if (!f) return 1;
  int n_seg, n_ticks, lag;
  double start[3], mc[18];
  if (fread(&n_seg, 4, 1, f) != 1) return 1;
  std::vector<double> coeffs(n_seg * 24), yaw0(n_seg);
  std::vector<int> rows(n_seg), table(n_seg);
  if (fread(coeffs.data(), 8, n_seg * 24, f) != (size_t)n_seg * 24) return 1;
  if (fread(rows.data(), 4, n_seg, f) != (size_t)n_seg) return 1;
  if (fread(table.data(), 4, n_seg, f) != (size_t)n_seg) return 1;
  if (fread(yaw0.data(), 8, n_seg, f) != (size_t)n_seg) return 1;
  if (fread(start, 8, 3, f) != 3) return 1;
  if (fread(&n_ticks, 4, 1, f) != 1) return 1;
  if (fread(&lag, 4, 1, f) != 1) return 1;
  if (fread(mc, 8, 18, f) != 18) return 1;   // mass scale, inertia scale[3], gain scale[11], wind[3]
  fclose(f);
  uavb_vehicle uv;
  vehicle_defaults(&uv);
  McValues o;
  o.mass = uv.mass * mc[0];
  for (int i = 0; i < 3; ++i) o.inertia[i] = uv.inertia[i] * mc[1 + i];
  for (int i = 0; i < 11; ++i) o.gains[i] = uv.gains[i] * mc[4 + i];
  for (int i = 0; i < 3; ++i) o.wind[i] = mc[15 + i];
  VehU<R> u;
  make_vehu<R>(u, uv, uv.dt * 10);
  VehP<R> v;
  make_vehp<R>(v, uv, o);
  MissionView m{coeffs.data(), rows.data(), table.data(), yaw0.data(), 0, n_seg, uv.dt * 10};
  Drone<R> d; Cursor<R> c; Accum<R> a;
  drone_init<R>(d, u, start[0], start[1], start[2]); cursor_init<R>(c); accum_init<R>(a);
  std::vector<double> log;
  VecLog<R> lg{&log, 10, 10};
  NoObstacles no;
  rollout_run<R>(d, c, a, u, v, m, 0, n_ticks, 10, lag, no, lg);
  FILE* g = fopen(outp, "wb");
  fwrite(log.data(), 8, log.size(), g);
  fclose(g);
  printf("periods %d mean_err %.9g rmse %.9g max %.9g status %d\n", a.periods, (double)a.sum_e / a.periods,
         sqrt((double)a.sum_e2 / a.periods), (double)a.max_e, a.status);
  return 0;
}

int main(int argc, char** argv) {
  if (argc < 4) return 2;
  return strcmp(argv[3], "f64") == 0 ? run<double>(argv[1], argv[2]) : run<float>(argv[1], argv[2]);
}
