// rollout_impl.cuh -- device side of K2 and its launchers, shared by the translation units that instantiate its kernels
// (two drones per thread, launch_pair: rollout_sliced.cu metrics only, rollout_log.cu state log, rollout_traj.cu flown-path list,
// rollout_tables.cu / rollout_tables_log.cu per-rollout caller tables; rollout_scalar.cu: one drone per thread for per-rollout
// missions; rollout_f64.cu: one-shot fp64 validation build).
//
// Each thread keeps its drone's 13-state, displacement accumulator, rotor speeds, controller integrator,
// commands, table cursor and metric accumulators in registers for a whole slice of the mission (hundreds to
// thousands of 1 kHz ticks), runs the cascade, allocation, motor lag and rigid-body step in fp32 every tick and
// touches memory only for
//   * its Monte-Carlo parameters (once per slice), the set-point row of the current outer period (56 bytes,
//     broadcast through L1 when the mission is shared; evaluated in fp64 from the staged spline otherwise),
//   * the optional state log [sample][field][B] (one streaming 4-byte store per field and thread: a warp writes
//     one full 128-byte line per field),
//   * the carry block between slices, metrics / final state at the end.
// Nothing here is a dense contraction, so no tensor-core path exists; the bound is the FP32 issue rate
// (metrics-only) or HBM (full-rate log).  See DESIGN.md "K2".
#pragma once

#include "rollout_core.cuh"
#include "rollout_pair.cuh"
#include "uavb_common.cuh"
#include "veh_setup.cuh"

namespace uavb {

// CTA shapes of the fp32 production rollout (two drones per thread, rollout_pair.cuh).  A pair needs ~200 registers, so the
// cap is 255 and an SM holds 8 warps = 512 drones -- the same number of drones in flight as the scalar kernel had with 16
// warps at 128 registers -- and two warps per scheduler fill the FMA pipe with packed instructions (measured,
// profiles/r02_ffma2_probe.md: 94 % at two independent chains per warp).
//   * metrics-only rollouts: ONE warp per CTA (64 drones), 8 CTAs per SM.  A work item ends with a CTA barrier, and with
//     per-rollout missions the warps of a CTA do different amounts of work (obstacle watching, rotor saturation): a second warp
//     only adds waiting at that barrier.
//   * rollouts with a state log: 64 threads (128 drones), 4 CTAs per SM -- a CTA writes 512 contiguous bytes per field and sample.
//   * fp64 validation build: one drone per thread, 64 threads, one-shot launch, 128 registers.
// 9 or 10 warps per SM at 224 / 208 / 192 registers and 12 at 168 measured slower (DESIGN.md, K2 round 2).
constexpr int kRolloutPairRegs = 255;
constexpr int kPairWarpsPerSm = 65536 / (32 * ((kRolloutPairRegs + 15) / 16 * 16));   // registers are allocated in units of 16 per thread
constexpr int kRolloutThreads = 32;
constexpr int kRolloutCtasPerSm = kPairWarpsPerSm;
constexpr int kRolloutThreadsLog = 64;
constexpr int kRolloutCtasPerSmLog = kPairWarpsPerSm / 2;
constexpr int kRolloutThreadsF64 = 64;
constexpr int kRolloutRegs = 128;          // fp64 validation build

template <class R> struct RolloutDev {
  uavb_rollout_args a;
  VehU<R> u;      // launch-uniform constants (constant bank)
  VehP<R> vp;     // per-rollout constants when no Monte-Carlo override is given (constant bank)
  int coeff_cache_offset;   // offset (in doubles) of the [24][64] coefficient staging area in dynamic shared memory, -1 = none
  // Sliced fp32 launches with Monte-Carlo overrides: the per-rollout constants (VehP) as [kVehpWords][vehp_stride] floats, written by a
  // pair's first slice and read by its later ones instead of redoing the ~20 fp64 divisions of make_vehp per drone and slice
  // (ncu: the slice prologue was half of the 10 us a slice costs the headline launch); nullptr = recompute.  Same values either way.
  float* vehp_cache;
  long long vehp_stride;
};

// Obstacle set: SHARED = one set for the launch, staged in the CTA's dynamic shared memory (LDS.64 broadcast reads);
// otherwise a per-rollout set in global memory.  A box is three (min, max) pairs; inclusive bounds exactly as
// is_collision_cuboid (minimum_snap.py:352-357).
template <bool SHARED> struct BoxesT {
  static constexpr bool kAny = true;
  const float* b;
  int n;
  __device__ __forceinline__ const float2* box(int i) const {
    if constexpr (SHARED) {
      extern __shared__ float2 s_box_pairs[];              // the same dynamic shared memory stage_shared_boxes fills
      return s_box_pairs + 3 * i;
    } else {
      return reinterpret_cast<const float2*>(b) + 3 * i;
    }
  }
  template <class R> __device__ __forceinline__ bool hit(R x, R y, R z) const {
    bool h = false;
    for (int i = 0; i < n; ++i) {
      const float2* q = box(i);
      const float2 bx = q[0], by = q[1], bz = q[2];
      h |= (bx.x <= x) & (x <= bx.y) & (by.x <= y) & (y <= by.y) & (bz.x <= z) & (z <= bz.y);
    }
    return h;
  }
  // Chebyshev gap from the point to the nearest box (<= 0 inside or on a face); NaN positions give NaN
  template <class R> __device__ __forceinline__ R gap(R x, R y, R z) const {
    R g = R(3.0e38);
    for (int i = 0; i < n; ++i) {
      const float2* q = box(i);
      const float2 bx = q[0], by = q[1], bz = q[2];
      const R gx = fmax((R)bx.x - x, x - (R)bx.y), gy = fmax((R)by.x - y, y - (R)by.y), gz = fmax((R)bz.x - z, z - (R)bz.y);
      const R gi = fmax(gx, fmax(gy, gz));
      g = (gi < g || gi != gi) ? gi : g;
    }
    return g;
  }
};

// [sample][13][B] state log, one sample after every `stride` ticks.
template <class R> struct GlobalLog {
  static constexpr bool kNormEveryTick = true;
  R* out;
  unsigned B;              // field stride in elements (check_args bounds 13 B below 2^32 when a log is requested)
  int stride, left;
  __device__ __forceinline__ void tick(const Drone<R>& d) {
    if (--left) return;
    left = stride;
    // streaming stores: the log is written once and never re-read by the kernel, keep it out of the L2 working set.
    // Field offsets are 32-bit multiples of B on one 64-bit base: cheaper address arithmetic than 64-bit products.
    R* o = out;
    const unsigned b = B;
    __stcs(o, (R)(d.px + (double)d.dx)); __stcs(o + (size_t)b, (R)(d.py + (double)d.dy)); __stcs(o + (size_t)(2u * b), (R)(d.pz + (double)d.dz));
    __stcs(o + (size_t)(3u * b), d.q0); __stcs(o + (size_t)(4u * b), d.q1); __stcs(o + (size_t)(5u * b), d.q2); __stcs(o + (size_t)(6u * b), d.q3);
    __stcs(o + (size_t)(7u * b), d.vx); __stcs(o + (size_t)(8u * b), d.vy); __stcs(o + (size_t)(9u * b), d.vz);
    __stcs(o + (size_t)(10u * b), d.wx); __stcs(o + (size_t)(11u * b), d.wy); __stcs(o + (size_t)(12u * b), d.wz);
    out = o + (size_t)(13u * b);
  }
};

__device__ __forceinline__ float i2f(int x) { return __int_as_float(x); }
__device__ __forceinline__ int f2i(float x) { return __float_as_int(x); }

// Resumable carry block, [UAVB_CARRY_WORDS][B] 32-bit words (fp32 rollout only).
struct Carry {
  float* p;
  long long B;
  __device__ __forceinline__ float& w(int k) const { return p[(long long)k * B]; }
  __device__ __forceinline__ void put64(int k, double x) const { w(k) = i2f(__double2loint(x)); w(k + 1) = i2f(__double2hiint(x)); }
  __device__ __forceinline__ double get64(int k) const { return __hiloint2double(f2i(w(k + 1)), f2i(w(k))); }
  __device__ void store(const Drone<float>& d, const Cursor<float>& c, const Accum<float>& a, int tick) const {
    put64(0, d.px); put64(2, d.py); put64(4, d.pz);
    w(6) = d.q0; w(7) = d.q1; w(8) = d.q2; w(9) = d.q3;
    w(10) = d.vx; w(11) = d.vy; w(12) = d.vz; w(13) = d.wx; w(14) = d.wy; w(15) = d.wz;
    w(16) = d.om0; w(17) = d.om1; w(18) = d.om2; w(19) = d.om3;
    w(20) = d.integral; w(21) = d.thrust_cmd; w(22) = d.cp; w(23) = d.cq; w(24) = d.cr;   // body-rate commands in rotor units
    w(25) = d.zbx; w(26) = d.zby; w(27) = d.zbz; w(28) = c.hx;
    w(29) = i2f(c.seg); w(30) = i2f(c.row); w(31) = i2f(c.phase);
    w(32) = c.ex; w(33) = c.ey; w(34) = c.ez;
    w(35) = 0.f; w(36) = 0.f; w(37) = 0.f;                  // spare
    w(38) = a.sum_e; w(39) = a.sum_e2; w(40) = a.max_e;
    w(41) = i2f(a.periods); w(42) = i2f(a.collided); w(43) = i2f(a.first_hit); w(44) = i2f(a.status);
    w(45) = i2f(tick);
    w(46) = d.dx; w(47) = d.dy; w(48) = d.dz; w(49) = c.hy;
  }
  __device__ void load(Drone<float>& d, Cursor<float>& c, Accum<float>& a, const VehU<float>& u, int* tick) const {
    d.px = get64(0); d.py = get64(2); d.pz = get64(4);
    d.q0 = w(6); d.q1 = w(7); d.q2 = w(8); d.q3 = w(9);
    d.vx = w(10); d.vy = w(11); d.vz = w(12); d.wx = w(13); d.wy = w(14); d.wz = w(15);
    d.om0 = w(16); d.om1 = w(17); d.om2 = w(18); d.om3 = w(19);
    d.integral = w(20); set_thrust_cmd<float>(d, u, w(21)); d.cp = w(22); d.cq = w(23); d.cr = w(24);
    d.zbx = w(25); d.zby = w(26); d.zbz = w(27); c.hx = w(28);
    c.seg = f2i(w(29)); c.row = f2i(w(30)); c.phase = f2i(w(31)); c.cached_seg = -1;
    c.ex = w(32); c.ey = w(33); c.ez = w(34);
    a.sum_e = w(38); a.sum_e2 = w(39); a.max_e = w(40);
    a.periods = f2i(w(41)); a.collided = f2i(w(42)); a.first_hit = f2i(w(43)); a.status = f2i(w(44));
    *tick = f2i(w(45));
    d.dx = w(46); d.dy = w(47); d.dz = w(48); c.hy = w(49);
  }
};

// Per-rollout constants of drone i (Monte-Carlo overrides applied).
template <class R> __device__ __forceinline__ void load_vehp(VehP<R>& v, const uavb_rollout_args& a, long long i) {
  const long long B = a.B;
  McValues mc;
  mc_from_vehicle(mc, a.veh);
  if (a.mc_mass) mc.mass = (double)a.mc_mass[i];
  if (a.mc_inertia) { mc.inertia[0] = (double)a.mc_inertia[i]; mc.inertia[1] = (double)a.mc_inertia[B + i]; mc.inertia[2] = (double)a.mc_inertia[2 * B + i]; }
  if (a.mc_gains) {
#pragma unroll
    for (int k = 0; k < UAVB_N_GAINS; ++k) mc.gains[k] = (double)a.mc_gains[k * B + i];
  }
  if (a.mc_wind) { mc.wind[0] = (double)a.mc_wind[i]; mc.wind[1] = (double)a.mc_wind[B + i]; mc.wind[2] = (double)a.mc_wind[2 * B + i]; }
  make_vehp<R>(v, a.veh, mc);
}

// The fields of VehP<float> in declaration order (the layout of RolloutDev::vehp_cache).
#define UAVB_VEHP_FIELDS(X)                                                                                                          \
  X(kf_dt_over_m) X(kf_dt_over_m2) X(dIx) X(dIy) X(dIz) X(Ikp_p) X(Ikp_q) X(Ikp_r) X(dt_invIx) X(dt_invIy) X(dt_invIz) X(Gx) X(Gy) X(Gz) \
  X(Jp) X(Jq) X(Jr) X(Wx) X(Wy) X(Wz) X(Kx) X(Ky) X(Kz) X(dvx) X(dvy) X(dvz) X(mass) X(kp_xy) X(kd_xy) X(kp_z) X(kd_z) X(ki_z)         \
  X(kp_roll) X(kp_pitch) X(kp_yaw) X(acc_max)
#define UAVB_COUNT_FIELD(f) +1
constexpr int kVehpWords = 0 UAVB_VEHP_FIELDS(UAVB_COUNT_FIELD);
static_assert(sizeof(VehP<float>) == 4 * kVehpWords, "UAVB_VEHP_FIELDS must list every field of VehP");
// column pair (2j, 2j+1) of the cache <-> the two VehP of a pair; fields the kernel never reads are never loaded
__device__ __forceinline__ void vehp_cache_store(float* cache, long long stride, long long i0, const VehP<float>& a, const VehP<float>& b) {
  float2* o = reinterpret_cast<float2*>(cache + i0);
  const long long s2 = stride >> 1;
  int k = 0;
#define UAVB_ST(f) o[(k++) * s2] = make_float2(a.f, b.f);
  UAVB_VEHP_FIELDS(UAVB_ST)
#undef UAVB_ST
}
__device__ __forceinline__ void vehp_cache_load(const float* cache, long long stride, long long i0, VehP<float>& a, VehP<float>& b) {
  const float2* o = reinterpret_cast<const float2*>(cache + i0);
  const long long s2 = stride >> 1;
  int k = 0;
#define UAVB_LD(f) { const float2 t = o[(k++) * s2]; a.f = t.x; b.f = t.y; }
  UAVB_VEHP_FIELDS(UAVB_LD)
#undef UAVB_LD
}

// The mission of drone i; `column` of `columns`: its column of the CTA's coefficient staging area (RolloutDev::coeff_cache_offset).
__device__ __forceinline__ void mission_view(MissionView& m, const uavb_rollout_args& a, int coeff_cache_offset, long long i, int column, int columns) {
  m.coeffs = a.seg_coeffs; m.rows = a.seg_rows; m.table = a.seg_table; m.yaw0 = a.seg_yaw0;
  m.seg_begin = a.mission_seg_begin ? a.mission_seg_begin[i] : 0;
  m.seg_count = a.mission_seg_count ? a.mission_seg_count[i] : a.n_seg_shared;
  m.dt_outer = a.dt_outer;
  m.trows = a.mission_seg_begin ? nullptr : static_cast<const TargetRow*>(a.shared_targets);
  m.n_trows = a.n_target_rows;
  m.cache = nullptr; m.cache_stride = 0;
  if (coeff_cache_offset >= 0) {               // on-the-fly evaluation: this drone's column of the CTA's coefficient staging area
    extern __shared__ double s_dyn_f64[];
    m.cache = s_dyn_f64 + coeff_cache_offset + column;
    m.cache_stride = columns;
  }
}

// Caller-supplied trajectory tables, one per rollout (uavb_rollout_tables_f32 with shared_rows = 0): rollout i flies the
// TargetRow records [offsets[t], offsets[t + 1]) of table t = table_index[i] (t = i when table_index is NULL).
struct TableSetDev {
  const TargetRow* rows;
  const long long* offsets;
  const int* table_index;
};

// The mission view of a per-rollout table: only trows / n_trows are read (PairTarget<kTargetPerRollout>); the cursor row is
// relative to the table, so the carry block resumes with the same table set.
__device__ __forceinline__ void table_view(MissionView& m, const TableSetDev& ts, long long i) {
  const long long t = ts.table_index ? (long long)ts.table_index[i] : i;
  const long long first = ts.offsets[t];
  m.coeffs = nullptr; m.rows = nullptr; m.table = nullptr; m.yaw0 = nullptr;
  m.seg_begin = 0; m.seg_count = 0; m.dt_outer = 0.0;
  m.trows = ts.rows + first;
  m.n_trows = (int)(ts.offsets[t + 1] - first);
  m.cache = nullptr; m.cache_stride = 0;
}

// Final outputs of one drone (state, metrics).  B: a.B, passed in so that drone_slice's one load of it serves the whole slice.
// log: the quaternion was renormalised in every tick (state-log bodies).
template <class R> __device__ __forceinline__ void write_outputs(const uavb_rollout_args& a, long long B, long long i, Drone<R>& d, const Cursor<R>& c,
                                                                const Accum<R>& acc, bool log) {
  const double fx = d.px + (double)d.dx, fy = d.py + (double)d.dy, fz = d.pz + (double)d.dz;
  if (a.state_out) {
    R* o = reinterpret_cast<R*>(a.state_out) + i;
    o[0 * B] = (R)fx; o[1 * B] = (R)fy; o[2 * B] = (R)fz;
    if (!log && c.phase != 0) renormalise_q<R>(d);           // the reported state is unit even in the middle of an outer period
    o[3 * B] = d.q0; o[4 * B] = d.q1; o[5 * B] = d.q2; o[6 * B] = d.q3;
    o[7 * B] = d.vx; o[8 * B] = d.vy; o[9 * B] = d.vz;
    o[10 * B] = d.wx; o[11 * B] = d.wy; o[12 * B] = d.wz;
  }
  if (a.metrics_out) {
    R fd = R(0);
    if (a.goal) {
      const double* g = a.goal + (size_t)a.goal_stride * i;
      const R ex = (R)(g[0] - fx), ey = (R)(g[1] - fy), ez = (R)(g[2] - fz);
      fd = Math<R>::sqrt(ex * ex + ey * ey + ez * ez);
    }
    const R np = acc.periods > 0 ? R(1) / (R)acc.periods : R(0);
    R* o = reinterpret_cast<R*>(a.metrics_out) + (size_t)i * UAVB_N_METRICS;
    o[UAVB_M_FINAL_DIST] = fd;
    o[UAVB_M_COLLISION] = (R)acc.collided;
    o[UAVB_M_RMSE] = Math<R>::sqrt(acc.sum_e2 * np);
    o[UAVB_M_MEAN_ERR] = acc.sum_e * np;
    o[UAVB_M_MAX_ERR] = acc.max_e;
    o[UAVB_M_STATUS] = (R)acc.status;
    o[UAVB_M_FIRST_HIT] = (R)acc.first_hit;
    o[UAVB_M_PERIODS] = (R)acc.periods;
  }
}

// One drone, one slice of its mission: `n_ticks` ticks starting from the carry block (from_carry) or from the start
// pose; writes the carry block (to_carry) and / or the final outputs (finish).
// MC: some per-rollout override (mass / inertia / gains / wind) is present; otherwise every vehicle constant is a
// constant-bank operand.
// `launch_tick0`: ticks of THIS launch that precede the slice (places the slice's samples in the state log).
template <class R, bool LOG, bool MC>
__device__ __forceinline__ void drone_slice(const RolloutDev<R>& p, long long i, int n_ticks, bool from_carry, bool to_carry, bool finish,
                                            int launch_tick0 = 0) {
  const uavb_rollout_args& a = p.a;
  const long long B = a.B;
  const bool shared_boxes = a.n_obs > 0 && a.aabb_set == nullptr;

  VehP<R> vloc;
  if constexpr (MC) load_vehp<R>(vloc, a, i);
  const VehP<R>& v = MC ? vloc : p.vp;
  const VehU<R>& u = p.u;

  MissionView m;
  mission_view(m, a, p.coeff_cache_offset, i, threadIdx.x, blockDim.x);

  Drone<R> d;
  Cursor<R> c;
  Accum<R> acc;
  int tick0 = 0;
  bool resumed = false;
  if constexpr (sizeof(R) == 4) {
    if (from_carry) {
      Carry cb{a.carry + i, B};
      cb.load(d, c, acc, u, &tick0);
      resumed = true;
    }
  }
  if (!resumed) {
    const double* s = a.start + (size_t)a.start_stride * i;
    drone_init<R>(d, u, s[0], s[1], s[2]);
    cursor_init<R>(c);
    accum_init<R>(acc);
  }

  auto fly = [&](const auto& obst) {
    if constexpr (LOG) {
      GlobalLog<R> lg;
      lg.out = reinterpret_cast<R*>(a.log_out) + (size_t)(launch_tick0 / a.log_stride) * 13 * B + i;
      lg.B = (unsigned)B; lg.stride = a.log_stride; lg.left = a.log_stride - launch_tick0 % a.log_stride;
      rollout_run<R>(d, c, acc, u, v, m, tick0, n_ticks, a.inner_per_outer, a.thrust_frame_lag, obst, lg, Ground{a.ground_on, a.ground_z});
    } else {
      NoLog lg;
      rollout_run<R>(d, c, acc, u, v, m, tick0, n_ticks, a.inner_per_outer, a.thrust_frame_lag, obst, lg, Ground{a.ground_on, a.ground_z});
    }
  };
  // three call sites, not four: the flying code is inlined at each (a floor without boxes is the shared set with n = 0 -- the
  // floor rides on the obstacle culling)
  if (a.n_obs > 0 && !shared_boxes) {
    fly(BoxesT<false>{a.aabbs + (size_t)a.aabb_set[i] * a.n_obs * 6, a.n_obs});
  } else if (a.n_obs > 0 || a.ground_on) {
    fly(BoxesT<true>{nullptr, a.n_obs});
  } else {
    fly(NoObstacles{});
  }

  if constexpr (sizeof(R) == 4) {
    if (to_carry) {
      Carry cb{a.carry + i, B};
      cb.store(d, c, acc, tick0 + n_ticks);
    }
  }
  if (finish) write_outputs(a, B, i, d, c, acc, LOG);
}

// One PAIR of drones (2j, 2j+1), one slice of their mission: the production fp32 path (rollout_pair.cuh).  Arguments as
// drone_slice.  When B is odd the last pair's second lane re-flies the first drone and writes nothing.
// LOG: 0 = no state log, 1 = per-thread streaming stores (PairLog), 2 = staged tensor stores (PairLogTma, `maps` required),
// 3 = the gated position list of the viewer (PairTrajLog; its state rides in the carry block between slices).
// MODE: where the set-points come from (kTargetFly / kTargetShared / kTargetPerRollout, rollout_pair.cuh); the last needs `tabs`.
template <int LOG, bool MC, int MODE, bool LAG>
__device__ __forceinline__ void pair_slice(const RolloutDev<float>& p, long long j, int n_ticks, bool from_carry, bool to_carry,
                                           bool finish, int launch_tick0, const LogTma* maps = nullptr, bool first_slice = true,
                                           const TableSetDev* tabs = nullptr, int spec_exact = 0) {
  const uavb_rollout_args& a = p.a;
  const long long B = a.B;
  const long long i0 = 2 * j;
  const bool second = i0 + 1 < B;
  const long long i1 = second ? i0 + 1 : i0;
  const bool shared_boxes = a.n_obs > 0 && a.aabb_set == nullptr;
  const VehU<float>& u = p.u;

  VehP<float> vloc[2];
  VehP2 v2;
  if constexpr (MC) {
    constexpr bool kCache = LOG != 3;                       // (the flown-path kernel has no register to spare for the two pointers)
    if (kCache && p.vehp_cache != nullptr && !first_slice) {   // (uniform) a later slice of a sliced launch: the constants its first slice made
      vehp_cache_load(p.vehp_cache, p.vehp_stride, i0, vloc[0], vloc[1]);
    } else {
      load_vehp<float>(vloc[0], a, i0);
      load_vehp<float>(vloc[1], a, i1);
      if (kCache && p.vehp_cache != nullptr) vehp_cache_store(p.vehp_cache, p.vehp_stride, i0, vloc[0], vloc[1]);
    }
    zip_vehp(v2, vloc[0], vloc[1]);
  }
  const VehP<float>& va = MC ? vloc[0] : p.vp;
  const VehP<float>& vb = MC ? vloc[1] : p.vp;
  VehO2 vo;
  zip_veho(vo, va, vb);

  MissionView ma, mb;
  if constexpr (MODE == kTargetPerRollout) {
    table_view(ma, *tabs, i0);
    table_view(mb, *tabs, i1);
  } else {
    mission_view(ma, a, p.coeff_cache_offset, i0, 2 * (int)threadIdx.x, 2 * (int)blockDim.x);
    mission_view(mb, a, p.coeff_cache_offset, i1, 2 * (int)threadIdx.x + 1, 2 * (int)blockDim.x);
  }

  Drone2 d;
  Cursor<float> c[2];
  Accum<float> acc[2];
  int tick0 = 0;
  if (from_carry) {
    Drone<float> s;
    Carry{a.carry + i0, B}.load(s, c[0], acc[0], u, &tick0);
    put_lane<0>(d, s, u);
    Carry{a.carry + i1, B}.load(s, c[1], acc[1], u, &tick0);
    put_lane<1>(d, s, u);
  } else {
    Drone<float> s;
    const double* s0 = a.start + (size_t)a.start_stride * i0;
    drone_init<float>(s, u, s0[0], s0[1], s0[2]);
    put_lane<0>(d, s, u);
    const double* s1 = a.start + (size_t)a.start_stride * i1;
    drone_init<float>(s, u, s1[0], s1[1], s1[2]);
    put_lane<1>(d, s, u);
    cursor_init<float>(c[0]); cursor_init<float>(c[1]);
    accum_init<float>(acc[0]); accum_init<float>(acc[1]);
  }

  double traj_time = 0.0, traj_next[2] = {0.0, 0.0};
  int traj_count[2] = {0, 0};
  auto fly = [&](const auto& oa, const auto& ob) {
    auto with_log = [&](auto& lg) {
      const Ground gr{a.ground_on, a.ground_z};
      if constexpr (kSpecBody<MODE, std::decay_t<decltype(lg)>>) {
        // speculative bodies: this thread's checkpoint slot after the staged boxes (launch_rollout sizes the area); made only here, so
        // that the other bodies compile to the same code as before
        const SpecSlot slot{(shared_boxes ? (24 * a.n_obs + 15) / 16 : 0) + (int)(threadIdx.x >> 5) * (32 * kSpecSlotVec4) + (int)(threadIdx.x & 31),
                            spec_exact};
        if constexpr (MC) rollout_run_pair<MODE, LAG>(d, c, acc, u, va, vb, v2, vo, ma, mb, tick0, n_ticks, a.inner_per_outer, oa, ob, lg, gr, slot);
        else rollout_run_pair<MODE, LAG>(d, c, acc, u, va, vb, p.vp, vo, ma, mb, tick0, n_ticks, a.inner_per_outer, oa, ob, lg, gr, slot);
      } else {
        if constexpr (MC) rollout_run_pair<MODE, LAG>(d, c, acc, u, va, vb, v2, vo, ma, mb, tick0, n_ticks, a.inner_per_outer, oa, ob, lg, gr);
        else rollout_run_pair<MODE, LAG>(d, c, acc, u, va, vb, p.vp, vo, ma, mb, tick0, n_ticks, a.inner_per_outer, oa, ob, lg, gr);
      }
    };
    if constexpr (LOG == 3) {
      PairTrajLog lg;
      lg.out = a.traj_out + i0; lg.B = B;
      lg.dt = a.veh.dt; lg.interval = a.traj_interval; lg.gate_z = a.traj_gate_z; lg.max_samples = a.traj_max_samples; lg.second = second;
      const Carry cb0{a.carry + i0, B}, cb1{a.carry + i1, B};
      if (from_carry) {                                    // words 35..37 / 50..51 of the carry block: next sample time, count / data.time
        lg.time = cb0.get64(50);
        lg.next[0] = cb0.get64(35); lg.count[0] = f2i(cb0.w(37));
        lg.next[1] = cb1.get64(35); lg.count[1] = f2i(cb1.w(37));
      } else {
        lg.time = 0.0; lg.next[0] = lg.next[1] = 0.0; lg.count[0] = lg.count[1] = 0;     // mujoco_sim.py:190-199
      }
      with_log(lg);
      traj_time = lg.time; traj_next[0] = lg.next[0]; traj_next[1] = lg.next[1]; traj_count[0] = lg.count[0]; traj_count[1] = lg.count[1];
    } else if constexpr (LOG == 2) {
      extern __shared__ __align__(128) float s_dyn_f32[];     // tensor stores read 128-byte aligned shared memory
      PairLogTma lg;
      lg.maps = maps;
      lg.stage = s_dyn_f32 + maps->stage_offset / 4 + (threadIdx.x >> 5) * kLogTmaWarpFloats;
      lg.mine = reinterpret_cast<float2*>(lg.stage) + (threadIdx.x & 31);
      lg.mask = __activemask();
      lg.col = (int)(2 * (j - (threadIdx.x & 31)));
      lg.sample = launch_tick0 / a.log_stride;
      lg.stride = a.log_stride; lg.left = a.log_stride - launch_tick0 % a.log_stride;
      lg.filled = 0; lg.buf = 0;
      with_log(lg);
      lg.finish();
    } else if constexpr (LOG == 1) {
      PairLog lg;
      lg.out = reinterpret_cast<float*>(a.log_out) + (size_t)(launch_tick0 / a.log_stride) * 13 * B + i0;
      lg.B = (unsigned)B; lg.stride = a.log_stride; lg.left = a.log_stride - launch_tick0 % a.log_stride;
      lg.vec = (B & 1) == 0; lg.second = second;
      with_log(lg);
    } else {
      NoPairLog lg;
      with_log(lg);
    }
  };
  // three call sites, not four: the flying code is inlined at each, and a fourth copy made ptxas keep the kernel parameter block
  // on the stack (a floor without boxes is the shared set with n = 0 -- the floor rides on the obstacle culling)
  if (a.n_obs > 0 && !shared_boxes) {
    fly(BoxesT<false>{a.aabbs + (size_t)a.aabb_set[i0] * a.n_obs * 6, a.n_obs}, BoxesT<false>{a.aabbs + (size_t)a.aabb_set[i1] * a.n_obs * 6, a.n_obs});
  } else if (a.n_obs > 0 || a.ground_on) {
    fly(BoxesT<true>{nullptr, a.n_obs}, BoxesT<true>{nullptr, a.n_obs});
  } else {
    fly(NoObstacles{}, NoObstacles{});
  }

  constexpr bool kStateLog = LOG == 1 || LOG == 2;          // per-tick quaternion normalisation
  Drone<float> s;
  get_lane<0>(d, s);
  if (to_carry) Carry{a.carry + i0, B}.store(s, c[0], acc[0], tick0 + n_ticks);
  if (finish) write_outputs(a, a.B, i0, s, c[0], acc[0], kStateLog);
  if (second) {
    get_lane<1>(d, s);
    if (to_carry) Carry{a.carry + i1, B}.store(s, c[1], acc[1], tick0 + n_ticks);
    if (finish) write_outputs(a, a.B, i1, s, c[1], acc[1], kStateLog);
  }
  if constexpr (LOG == 3) {
    if (to_carry) {
      const Carry cb0{a.carry + i0, B};
      cb0.put64(50, traj_time); cb0.put64(35, traj_next[0]); cb0.w(37) = i2f(traj_count[0]);
      if (second) {
        const Carry cb1{a.carry + i1, B};
        cb1.put64(50, traj_time); cb1.put64(35, traj_next[1]); cb1.w(37) = i2f(traj_count[1]);
      }
    }
    if (finish && a.traj_count_out) {
      a.traj_count_out[i0] = traj_count[0];
      if (second) a.traj_count_out[i1] = traj_count[1];
    }
  }
}

__device__ __forceinline__ void stage_shared_boxes(const uavb_rollout_args& a, float* s_boxes) {
  if (a.n_obs > 0 && a.aabb_set == nullptr) {
    for (int j = threadIdx.x; j < a.n_obs * 6; j += blockDim.x) s_boxes[j] = a.aabbs[j];
    __syncthreads();
  }
}

// One-shot launch: thread i flies drone i for the whole launch (the fp64 validation build).
template <class R, bool LOG, bool MC>
__global__ void __maxnreg__(kRolloutRegs) rollout_kernel(const __grid_constant__ RolloutDev<R> p) {
  extern __shared__ float s_boxes[];
  stage_shared_boxes(p.a, s_boxes);
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.a.B) return;
  drone_slice<R, LOG, MC>(p, i, p.a.n_ticks, p.a.resume != 0, p.a.carry != nullptr, true);
}

// Time-sliced persistent launch (every fp32 rollout, with or without a state log).  When the batch needs between one and a few waves of
// CTAs, a one-shot launch ends with a long tail: every CTA lives for the whole mission, so the last partial wave costs a full
// mission time at a fraction of the machine.  Here the grid is exactly the resident capacity, the mission is cut into
// `n_chunks` slices of `chunk_ticks` ticks, and CTAs pull (chunk, group) items from an atomic counter in chunk-major
// order; between slices a drone's state rests in the carry block (208 B per drone and slice, ~0.2 B per tick).  Item
// (c, g) needs (c-1, g), which was handed out one full sweep of the groups earlier, so the wait on its completion flag
// practically never spins -- and cannot deadlock, because whoever holds the earlier item is running.  The tail shrinks
// from one mission to one slice.
constexpr int kSliceTab = 64;
struct SliceSched {
  int* counter;        // next item
  int* done;           // [n_groups] slices completed per group
  int n_groups, n_chunks, chunk_ticks;
  int final_carry;     // the caller asked for the carry block of the end state
  int n_tab;           // > 0: slice c covers ticks [tab[c], tab[c + 1]) (n_chunks <= kSliceTab slices of unequal length); 0: c * chunk_ticks
  int tab[kSliceTab + 1];
  __device__ __forceinline__ int begin(int c) const { return n_tab ? tab[c] : c * chunk_ticks; }
};

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) { asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

// The work-item loop of a persistent launch.  A thread flies PER drones (1: drone k, 2: the pair 2k, 2k+1) of its CTA's work group; for
// every (chunk, group) item the CTA pulls it runs item(k, chunk, t0, ticks, last) -- `ticks` ticks from launch tick t0, `last`: the final
// slice -- once the group's previous slice has completed, and publishes the item's completion.
template <int PER, class F> __device__ __forceinline__ void slice_items(const uavb_rollout_args& a, const SliceSched& sch, F&& item) {
  __shared__ int s_item;
  const int n_items = sch.n_groups * sch.n_chunks;
  for (;;) {
    if (threadIdx.x == 0) {
      const int it = atomicAdd(sch.counter, 1);
      if (it < n_items) {
        const int c = it / sch.n_groups, g = it - c * sch.n_groups;
        while (ld_acquire_gpu(sch.done + g) < c) __nanosleep(200);
      }
      s_item = it;
    }
    __syncthreads();
    const int it = s_item;
    if (it >= n_items) return;
    const int c = it / sch.n_groups, g = it - c * sch.n_groups;
    const long long k = (long long)g * blockDim.x + threadIdx.x;
    if (PER * k < a.B) {
      const bool last = c == sch.n_chunks - 1;
      const int t0 = sch.begin(c);
      const int ticks = last ? a.n_ticks - t0 : sch.begin(c + 1) - t0;
      item(k, c, t0, ticks, last);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) st_release_gpu(sch.done + g, c + 1);
  }
}

template <bool MC, int MODE, int LOG, bool LAG>
__device__ __forceinline__ void sliced_body(const RolloutDev<float>& p, const SliceSched& sch, const LogTma* maps, const TableSetDev* tabs = nullptr,
                                            int spec_exact = 0) {
  extern __shared__ __align__(128) float s_boxes[];
  stage_shared_boxes(p.a, s_boxes);
  slice_items<2>(p.a, sch, [&](long long j, int c, int t0, int ticks, bool last) {
    pair_slice<LOG, MC, MODE, LAG>(p, j, ticks, c > 0 || p.a.resume != 0, !last || sch.final_carry != 0, last, t0, maps, c == 0, tabs, spec_exact);
  });
}

// spec_exact: development switch of the speculative bodies (uavb_dev_speculation), read by the metrics-only table bodies only
template <bool MC, bool TABLE, bool LOG, bool LAG>
__global__ void __maxnreg__(kRolloutPairRegs) rollout_sliced_kernel(const __grid_constant__ RolloutDev<float> p, const SliceSched sch, int spec_exact) {
  sliced_body<MC, TABLE ? kTargetShared : kTargetFly, LOG ? 1 : 0, LAG>(p, sch, nullptr, nullptr, spec_exact);
}

// One drone per thread at 128 registers, 16 one-warp CTAs per SM: the round-1 kernel, kept for metrics-only rollouts with PER-ROLLOUT
// missions.  There the warps of an SM sit at different phases (own splines, own obstacle sets, rotor limits in most ticks), the
// fp64 set-point evaluation is inlined once instead of twice, and four warps per scheduler hide what two cannot: measured 98 ms
// against 108 ms for the pair kernel on BASELINE configs[3].
constexpr int kScalarThreads = 32;
constexpr int kScalarCtasPerSm = 16;
template <bool MC>
__global__ void __maxnreg__(kRolloutRegs) rollout_sliced_scalar_kernel(const __grid_constant__ RolloutDev<float> p, const SliceSched sch) {
  extern __shared__ __align__(128) float s_boxes[];
  stage_shared_boxes(p.a, s_boxes);
  slice_items<1>(p.a, sch, [&](long long i, int c, int t0, int ticks, bool last) {
    drone_slice<float, false, MC>(p, i, ticks, c > 0 || p.a.resume != 0, !last || sch.final_carry != 0, last, t0);
  });
}

// Metrics + the gated position list of the viewer (PairTrajLog); one-warp CTAs like the metrics-only kernel.
template <bool MC, bool TABLE, bool LAG>
__global__ void __maxnreg__(kRolloutPairRegs) rollout_sliced_traj_kernel(const __grid_constant__ RolloutDev<float> p, const SliceSched sch) {
  sliced_body<MC, TABLE ? kTargetShared : kTargetFly, 3, LAG>(p, sch, nullptr);
}

// The state log through staged tensor stores (PairLogTma); `maps` lives in the kernel parameter space, where the TMA unit reads it.
template <bool MC, bool TABLE, bool LAG>
__global__ void __maxnreg__(kRolloutPairRegs) rollout_sliced_tma_kernel(const __grid_constant__ RolloutDev<float> p, const SliceSched sch,
                                                                         const __grid_constant__ LogTma maps) {
  sliced_body<MC, TABLE ? kTargetShared : kTargetFly, 2, LAG>(p, sch, &maps);
}

// The same three families flying caller-supplied tables, one per rollout (kTargetPerRollout): metrics only or per-thread log
// stores, the flown-path list, staged tensor stores.  `ts` lives in the kernel parameter space like `maps`.
template <bool MC, bool LOG, bool LAG>
__global__ void __maxnreg__(kRolloutPairRegs) rollout_sliced_tables_kernel(const __grid_constant__ RolloutDev<float> p, const SliceSched sch,
                                                                            const __grid_constant__ TableSetDev ts, int spec_exact) {
  sliced_body<MC, kTargetPerRollout, LOG ? 1 : 0, LAG>(p, sch, nullptr, &ts, spec_exact);
}
template <bool MC, bool LAG>
__global__ void __maxnreg__(kRolloutPairRegs) rollout_sliced_tables_traj_kernel(const __grid_constant__ RolloutDev<float> p, const SliceSched sch,
                                                                                 const __grid_constant__ TableSetDev ts) {
  sliced_body<MC, kTargetPerRollout, 3, LAG>(p, sch, nullptr, &ts);
}
template <bool MC, bool LAG>
__global__ void __maxnreg__(kRolloutPairRegs) rollout_sliced_tables_tma_kernel(const __grid_constant__ RolloutDev<float> p, const SliceSched sch,
                                                                                const __grid_constant__ LogTma maps, const __grid_constant__ TableSetDev ts) {
  sliced_body<MC, kTargetPerRollout, 2, LAG>(p, sch, &maps, &ts);
}


// Development switch of the speculative bodies (rollout_pair.cuh, set by uavb_dev_speculation): fly every stretch exactly.
extern int g_spec_exact;

// Launch of a pair kernel: MODE (kTargetFly / kTargetShared / kTargetPerRollout, `ts` required for the last) and LOG (as pair_slice;
// 2 requires `maps`) pick the kernel family and its CTA shape, mc and lag its instantiation.  Each (MODE, LOG) is instantiated by the
// translation unit that compiles its kernels (UAVB_LAUNCH_PAIR below), so that the units compile in parallel.
template <int MODE, int LOG>
void launch_pair(bool mc, bool lag, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch, const LogTma* maps,
                 const TableSetDev* ts) {
  constexpr int threads = (LOG == 1 || LOG == 2) ? kRolloutThreadsLog : kRolloutThreads;
  auto go = [&](auto mc_c, auto lag_c) {
    constexpr bool MC = decltype(mc_c)::value, LAG = decltype(lag_c)::value;
    if constexpr (MODE == kTargetPerRollout) {
      if constexpr (LOG == 3) rollout_sliced_tables_traj_kernel<MC, LAG><<<grid, threads, smem, st>>>(p, sch, *ts);
      else if constexpr (LOG == 2) rollout_sliced_tables_tma_kernel<MC, LAG><<<grid, threads, smem, st>>>(p, sch, *maps, *ts);
      else rollout_sliced_tables_kernel<MC, LOG == 1, LAG><<<grid, threads, smem, st>>>(p, sch, *ts, g_spec_exact);
    } else {
      constexpr bool TABLE = MODE == kTargetShared;
      if constexpr (LOG == 3) rollout_sliced_traj_kernel<MC, TABLE, LAG><<<grid, threads, smem, st>>>(p, sch);
      else if constexpr (LOG == 2) rollout_sliced_tma_kernel<MC, TABLE, LAG><<<grid, threads, smem, st>>>(p, sch, *maps);
      else rollout_sliced_kernel<MC, TABLE, LOG == 1, LAG><<<grid, threads, smem, st>>>(p, sch, g_spec_exact);
    }
  };
  if (mc) {
    if (lag) go(BoolC<true>{}, BoolC<true>{}); else go(BoolC<true>{}, BoolC<false>{});
  } else {
    if (lag) go(BoolC<false>{}, BoolC<true>{}); else go(BoolC<false>{}, BoolC<false>{});
  }
}
#define UAVB_LAUNCH_PAIR(MODE, LOG)                                                                                                  \
  template void launch_pair<MODE, LOG>(bool, bool, int, size_t, cudaStream_t, const RolloutDev<float>&, const SliceSched&, const LogTma*, \
                                       const TableSetDev*)
extern UAVB_LAUNCH_PAIR(kTargetFly, 0); extern UAVB_LAUNCH_PAIR(kTargetFly, 1); extern UAVB_LAUNCH_PAIR(kTargetFly, 2); extern UAVB_LAUNCH_PAIR(kTargetFly, 3);
extern UAVB_LAUNCH_PAIR(kTargetShared, 0); extern UAVB_LAUNCH_PAIR(kTargetShared, 1); extern UAVB_LAUNCH_PAIR(kTargetShared, 2);
extern UAVB_LAUNCH_PAIR(kTargetShared, 3);
extern UAVB_LAUNCH_PAIR(kTargetPerRollout, 0); extern UAVB_LAUNCH_PAIR(kTargetPerRollout, 1); extern UAVB_LAUNCH_PAIR(kTargetPerRollout, 2);
extern UAVB_LAUNCH_PAIR(kTargetPerRollout, 3);

void launch_rollout_sliced_scalar(bool mc, int grid, size_t smem, cudaStream_t st, const RolloutDev<float>& p, const SliceSched& sch);
void launch_rollout_f64(bool log, bool mc, int grid, size_t smem, cudaStream_t st, const RolloutDev<double>& p);

}  // namespace uavb
