// rollout_kernels.cu -- K2 host side: argument checks, launch policy (time slicing, scratch), the set-point table of a
// shared mission, and the C entry points.  The device code lives in rollout_impl.cuh; its kernels are instantiated, with their
// launchers, in rollout_sliced.cu / rollout_log.cu / rollout_traj.cu / rollout_tables.cu / rollout_tables_log.cu (two drones per
// thread), rollout_scalar.cu (one drone per thread) and rollout_f64.cu (fp64 validation build).
#include "rollout_impl.cuh"

namespace uavb {

int g_spec_exact = 0;

// ---------------------------------------------------------------------------------------------
// Set-point table of a shared mission.  Pass 1 (one thread per row): polynomial values and the row's own heading
// (velocity direction where the horizontal speed reaches the threshold, NaN elsewhere).  Pass 2: every row takes the
// heading of the last valid row at or before it inside its MinimumSnap table, or the table's look-ahead yaw when there is
// none -- exactly the values cursor_target carries from row to row.
__global__ void __launch_bounds__(128) target_rows_kernel(const double* __restrict__ coeffs, const int* __restrict__ rows,
                                                          const int* __restrict__ table, int n_seg, double dt_outer,
                                                          TargetRow* __restrict__ out, float2* __restrict__ raw, int* __restrict__ tstart,
                                                          int n_rows) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_rows) return;
  int seg = 0, first = 0, tab_first = 0;                    // segment of row g, its first row, first row of its table
  int last_seg = 0, last_first = 0, last_tab = 0;            // last segment that owns rows (for rows past the end of the mission)
  for (; seg < n_seg; ++seg) {
    if (table[seg]) tab_first = first;
    if (rows[seg] > 0) { last_seg = seg; last_first = first; last_tab = tab_first; }
    if (g < first + rows[seg]) break;
    first += rows[seg];
  }
  int local = g - first;
  if (seg == n_seg) { seg = last_seg; first = last_first; tab_first = last_tab; local = rows[seg] - 1; }   // hold the last row (main.py:61)
  const double* cf = coeffs + (size_t)seg * 24;
  double p[3], v[3], a[3];
  eval_row([cf](int i) { return __ldg(cf + i); }, (double)local * dt_outer, p, v, a);
  TargetRow r;
  r.x = p[0]; r.y = p[1]; r.z = p[2];
  r.vx = (float)v[0]; r.vy = (float)v[1]; r.vz = (float)v[2];
  r.ax = (float)a[0]; r.ay = (float)a[1]; r.az = (float)a[2];
  r.yc = 0.f; r.ys = 0.f;
  out[g] = r;
  const bool valid = speed2_unfused(v[0], v[1]) >= kSpeed2Min;
  raw[g] = valid ? make_float2((float)v[0], (float)v[1]) : make_float2(nanf(""), nanf(""));
  tstart[g] = (tab_first << 8) | seg;                       // n_seg <= 2 * UAVB_MAX_SPLINES < 256
}

__global__ void __launch_bounds__(128) target_heading_kernel(const float2* __restrict__ raw, const int* __restrict__ tstart,
                                                             const double* __restrict__ yaw0, const int* __restrict__ rows, int n_seg,
                                                             TargetRow* __restrict__ out, int n_rows) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_rows) return;
  const int tab_first = tstart[g] >> 8;
  int r = g;
  float2 h = raw[r];
  while (h.x != h.x && r > tab_first) h = raw[--r];
  if (h.x != h.x) {                                         // no valid row yet in this table: its look-ahead yaw
    int seg = 0, first = 0;
    while (seg < n_seg && first != tab_first) first += rows[seg++];
    const double y0 = yaw0[seg];
    h = make_float2((float)cos(y0), (float)sin(y0));
  }
  out[g].yc = h.x; out[g].ys = h.y;
}

// tables: the arguments of uavb_rollout_tables_f32, where the set-points come from a uavb_table_set and every mission-segment field
// must be NULL / 0.
static int check_args(const uavb_rollout_args* a, bool f64, bool tables = false) {
  UAVB_REQUIRE(a != nullptr, "rollout: args is NULL");
  UAVB_REQUIRE(a->B >= 0 && a->n_ticks >= 0, "rollout: B and n_ticks must be >= 0");
  UAVB_REQUIRE(a->inner_per_outer >= 1, "rollout: inner_per_outer must be >= 1");
  if (tables) {
    UAVB_REQUIRE(!a->seg_coeffs && !a->seg_rows && !a->seg_table && !a->seg_yaw0 && !a->mission_seg_begin && !a->mission_seg_count &&
                     a->n_seg_shared == 0 && !a->shared_targets && a->n_target_rows == 0,
                 "rollout_tables: the mission-segment fields of args (seg_*, mission_seg_*, n_seg_shared, shared_targets, n_target_rows) "
                 "must be NULL / 0");
  } else {
    UAVB_REQUIRE(a->seg_coeffs && a->seg_rows && a->seg_table && a->seg_yaw0, "rollout: mission segment arrays are required");
    UAVB_REQUIRE((a->mission_seg_begin == nullptr) == (a->mission_seg_count == nullptr),
                 "rollout: mission_seg_begin and mission_seg_count must be given together");
    UAVB_REQUIRE(a->mission_seg_begin != nullptr || a->n_seg_shared >= 1, "rollout: n_seg_shared must be >= 1 for a shared mission");
  }
  UAVB_REQUIRE(a->resume || a->start != nullptr, "rollout: start is required when resume = 0");
  UAVB_REQUIRE(a->start_stride == 0 || a->start_stride == 3, "rollout: start_stride must be 0 or 3");
  UAVB_REQUIRE(a->goal == nullptr || a->goal_stride == 0 || a->goal_stride == 3, "rollout: goal_stride must be 0 or 3");
  UAVB_REQUIRE(!a->resume || a->carry != nullptr, "rollout: resume = 1 needs a carry block");
  UAVB_REQUIRE(!(f64 && (a->resume || a->carry)), "rollout_f64: the fp64 validation rollout has no carry/resume");
  UAVB_REQUIRE(a->log_stride >= 0, "rollout: log_stride must be >= 0");
  UAVB_REQUIRE(a->n_slices >= 0, "rollout: n_slices must be >= 0");
  UAVB_REQUIRE(a->log_stride == 0 || a->log_out != nullptr, "rollout: log_stride > 0 needs log_out");
  UAVB_REQUIRE(a->log_stride == 0 || a->B <= 300000000LL, "rollout: a state log supports at most 3e8 rollouts per launch");
  UAVB_REQUIRE(a->traj_out == nullptr || (!f64 && a->log_stride == 0), "rollout: traj_out is for fp32 rollouts without a state log");
  UAVB_REQUIRE(a->traj_out == nullptr || (a->traj_max_samples >= 1 && a->traj_interval >= 0.0), "rollout: traj_out needs traj_max_samples >= 1 and traj_interval >= 0");
  UAVB_REQUIRE(a->n_obs >= 0 && a->n_obs <= 1024, "rollout: n_obs out of range");
  UAVB_REQUIRE(a->n_obs == 0 || (a->aabbs != nullptr && a->n_obs_sets >= 1), "rollout: n_obs > 0 needs aabbs and n_obs_sets >= 1");
  UAVB_REQUIRE((tables || a->dt_outer > 0.0) && a->veh.dt > 0.0 && a->veh.mass > 0.0, "rollout: dt_outer, veh.dt and veh.mass must be positive");
  UAVB_REQUIRE(a->shared_targets == nullptr || (a->mission_seg_begin == nullptr && a->n_target_rows >= 1),
               "rollout: shared_targets needs a shared mission and n_target_rows >= 1");
  return UAVB_OK;
}

// Stream-ordered scratch that frees itself when the launcher returns (the free is ordered after the kernel).
struct StreamScratch {
  cudaStream_t st;
  void* p = nullptr;
  explicit StreamScratch(cudaStream_t s) : st(s) {}
  ~StreamScratch() { if (p) cudaFreeAsync(p, st); }
  cudaError_t alloc(size_t bytes) {
    cudaMemPool_t pool = scratch_pool();
    return pool ? cudaMallocFromPoolAsync(&p, bytes, pool, st) : cudaMallocAsync(&p, bytes, st);
  }
};

// tabs != nullptr: per-rollout caller tables (fp32 only).  checked: the caller validated the arguments (uavb_rollout_tables_f32).
template <class R> static int launch_rollout(const uavb_rollout_args* a, void* stream, const TableSetDev* tabs = nullptr, bool checked = false) {
  int rc = checked ? UAVB_OK : check_args(a, sizeof(R) == 8);
  if (rc) return rc;
  rc = require_device();
  if (rc) return rc;
  if (a->B == 0) return UAVB_OK;
  RolloutDev<R> p;
  p.a = *a;
  make_vehu<R>(p.u, a->veh, a->dt_outer);
  McValues mc;
  mc_from_vehicle(mc, a->veh);
  make_vehp<R>(p.vp, a->veh, mc);
  const bool log = a->log_stride > 0;
  // fp32 metrics-only rollouts with per-rollout missions fly one drone per thread (rollout_sliced_scalar_kernel), everything else in fp32 a pair
  const bool scalar32 = sizeof(R) == 4 && !log && a->traj_out == nullptr && a->mission_seg_begin != nullptr && a->pair_kernel_only == 0;
  const int threads = sizeof(R) == 8 ? kRolloutThreadsF64 : (log ? kRolloutThreadsLog : (scalar32 ? kScalarThreads : kRolloutThreads));
  // fp32: a thread flies a PAIR of drones (rollout_pair.cuh), so a CTA (= one work group of the slice scheduler) covers 2 x threads
  const int per_cta = (sizeof(R) == 8 || scalar32) ? threads : 2 * threads;
  const int grid = div_up(a->B, per_cta);
  size_t smem = (a->n_obs > 0 && a->aabb_set == nullptr) ? sizeof(float) * 6 * a->n_obs : 0;
  p.coeff_cache_offset = -1;
  p.vehp_cache = nullptr;
  p.vehp_stride = 0;
  const bool from_table = a->shared_targets != nullptr && a->mission_seg_begin == nullptr;
  if (!from_table && tabs == nullptr && sizeof(R) == 4) {                            // fp32 kernels stage the current spline in shared memory
    smem = (smem + 7) / 8 * 8;
    p.coeff_cache_offset = (int)(smem / 8);
    smem += sizeof(double) * 24 * per_cta;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool mc_any = a->mc_mass || a->mc_inertia || a->mc_gains || a->mc_wind;
  if constexpr (sizeof(R) == 8) {                      // validation build
    (void)tabs;
    launch_rollout_f64(log, mc_any, grid, smem, st, p);
  } else {
    int sms = 0;
    rc = sm_count_cached(&sms);
    if (rc) return rc;
    // fp32 launches ALWAYS run the time-sliced persistent kernel (16 warps per SM at 128 registers, CTA shapes in rollout_impl.cuh), with a single
    // slice when slicing has nothing to gain; a state log is written slice by slice into its place.  One compiled body for every batch size keeps
    // per-rollout results independent of how a job is sharded (ptxas fuses mul+add differently under different register
    // caps, so differently compiled variants are NOT bit-identical to each other).
    const int slots = sms * (log ? kRolloutCtasPerSmLog : (scalar32 ? kScalarCtasPerSm : kRolloutCtasPerSm));
    // ~32 items per resident CTA keep the tail near 3 % of the launch; slices are whole outer periods of >= 100 ticks
    constexpr int kMinChunkTicks = 100;
    long long want = grid > slots ? (32LL * slots + grid - 1) / grid : 1;
    if (a->n_slices > 0) want = a->n_slices < 4096 ? a->n_slices : 4096;         // uavb.h: results are independent of the slice count
    const int period = a->inner_per_outer;
    int chunk = (int)((a->n_ticks + want - 1) / want);
    chunk = ((chunk + period - 1) / period) * period;
    if (chunk < kMinChunkTicks) chunk = ((kMinChunkTicks + period - 1) / period) * period;
    const int n_chunks = a->n_ticks > 0 ? (a->n_ticks + chunk - 1) / chunk : 1;
    StreamScratch flags(st), carry(st), consts(st);
    const size_t n_flags = (size_t)grid + 1;
    cudaError_t e = flags.alloc(n_flags * sizeof(int));
    if (e == cudaSuccess) e = cudaMemsetAsync(flags.p, 0, n_flags * sizeof(int), st);
    SliceSched sch;
    sch.final_carry = a->carry != nullptr;
    if (e == cudaSuccess && a->carry == nullptr && n_chunks > 1) {
      e = carry.alloc(sizeof(float) * UAVB_CARRY_WORDS * (size_t)a->B);
      p.a.carry = static_cast<float*>(carry.p);
    }
    if (e == cudaSuccess && mc_any && n_chunks > 1 && !scalar32) {      // the pairs' per-rollout constants, made by slice 0 (rollout_impl.cuh)
      const long long padded = 2LL * div_up(a->B, 2);
      e = consts.alloc(sizeof(float) * kVehpWords * (size_t)padded);
      p.vehp_cache = static_cast<float*>(consts.p);
      p.vehp_stride = padded;
    }
    if (e != cudaSuccess) {
      cudaGetLastError();
      return set_error(UAVB_ENOMEM, "rollout: scratch allocation failed: %s", cudaGetErrorString(e));
    }
    sch.counter = static_cast<int*>(flags.p);
    sch.done = sch.counter + 1;
    sch.n_groups = grid; sch.n_chunks = n_chunks; sch.chunk_ticks = chunk;
    sch.n_tab = 0;
    // Slices of DECREASING length (unless the caller forces a slice count): every slice costs a carry round trip
    // (~5 us per 1e5 rollouts), the tail of the launch is one slice of the last kind long -- so each slice takes a fifth of what is left
    // (whole outer periods), down to a length that is <= 0.5 % of a resident CTA's share of the launch and >= 200 ticks.  Measured on the
    // headline launch (1e5 x 10 760 ticks, 1 563 groups on 1 184 resident CTAs): 15 such slices 4.605 ms against 4.653 ms for the 25 equal
    // slices of the rule above (tools/pipeline_probe.py).  Results do not depend on the slicing (tests/test_rollout_gpu.py).
    // The two constants sit on a flat optimum: fractions 1/3 ... 1/8 with floors of 100 ... 400 ticks land within +-0.7 % (DESIGN.md).
    constexpr int kSlicePart = 5, kSliceFloorTicks = 200;
    if (a->n_slices <= 0 && n_chunks > 1) {
      const double share = (double)grid / (double)slots * (double)a->n_ticks;       // ticks a resident CTA flies in this launch
      int min_len = share / 200.0 < (double)a->n_ticks ? (int)(share / 200.0) : a->n_ticks;     // (never longer than the launch: no overflow below)
      if (min_len < kSliceFloorTicks) min_len = kSliceFloorTicks;
      min_len = (int)(((long long)min_len + period - 1) / period * period);
      int t = 0, n = 0;
      sch.tab[0] = 0;
      while (t < a->n_ticks) {
        const int left = a->n_ticks - t;
        int len = left / kSlicePart;
        if (len < min_len) len = min_len;
        const long long whole = ((long long)len + period - 1) / period * period;      // whole outer periods
        len = whole < left ? (int)whole : left;
        if (n == kSliceTab - 1) len = left;
        if (left - len < min_len / 2) len = left;                                    // no sliver at the end
        t += len;
        sch.tab[++n] = t;
      }
      sch.n_tab = n; sch.n_chunks = n;
    }
    // metrics-only shared-table / per-rollout-table bodies: the speculative stretches' checkpoints (rollout_pair.cuh), 160 B per thread
    // after the staged boxes -- 5 KB per one-warp CTA, 8 CTAs per SM stay resident
    if (!log && a->traj_out == nullptr && !scalar32 && (from_table || tabs)) {
      smem = (smem + 15) / 16 * 16;
      smem += sizeof(float4) * kSpecSlotVec4 * threads;
    }
    const int pgrid = slots < grid ? slots : grid;
    // state log: through the TMA unit when the [samples x 13][B] log is a legal tensor (rows a multiple of 16 bytes, 16-byte aligned)
    LogTma maps;
    bool tma_log = false;
    if (log && a->log_tma >= 0) {
      const unsigned long long n_samples = (unsigned long long)(a->n_ticks / a->log_stride);
      if (a->B % 4 == 0 && n_samples > 0 && n_samples * 13ull < 2000000000ull) {
        tma_log = make_tensor_map_2d(&maps.box_k, a->log_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (unsigned long long)a->B, n_samples * 13ull, 4ull * a->B, 64,
                                     13 * kLogTmaSamples, CU_TENSOR_MAP_SWIZZLE_NONE) &&
                  make_tensor_map_2d(&maps.box_1, a->log_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (unsigned long long)a->B, n_samples * 13ull, 4ull * a->B, 64, 13,
                                     CU_TENSOR_MAP_SWIZZLE_NONE);
      }
      if (tma_log) {
        smem = (smem + 127) / 128 * 128;
        maps.stage_offset = (int)smem;
        smem += sizeof(float) * kLogTmaWarpFloats * (kRolloutThreadsLog / 32);
      }
    }
    const RolloutDev<float>& p32 = *reinterpret_cast<RolloutDev<float>*>(&p);
    if (scalar32) {
      launch_rollout_sliced_scalar(mc_any, pgrid, smem, st, p32, sch);
    } else {
      typedef void (*PairLaunch)(bool, bool, int, size_t, cudaStream_t, const RolloutDev<float>&, const SliceSched&, const LogTma*, const TableSetDev*);
      static constexpr PairLaunch kPairLaunch[3][4] = {
          {launch_pair<kTargetFly, 0>, launch_pair<kTargetFly, 1>, launch_pair<kTargetFly, 2>, launch_pair<kTargetFly, 3>},
          {launch_pair<kTargetShared, 0>, launch_pair<kTargetShared, 1>, launch_pair<kTargetShared, 2>, launch_pair<kTargetShared, 3>},
          {launch_pair<kTargetPerRollout, 0>, launch_pair<kTargetPerRollout, 1>, launch_pair<kTargetPerRollout, 2>, launch_pair<kTargetPerRollout, 3>}};
      const int mode = tabs ? kTargetPerRollout : from_table ? kTargetShared : kTargetFly;
      const int log_kind = log ? (tma_log ? 2 : 1) : a->traj_out ? 3 : 0;           // pair_slice's LOG
      kPairLaunch[mode][log_kind](mc_any, a->thrust_frame_lag != 0, pgrid, smem, st, p32, sch, tma_log ? &maps : nullptr, tabs);
    }
  }
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

// Caller tables -> set-point rows (uavb_table_targets_f64), one thread per row: x y z copied, v / a rounded once to fp32, the yaw
// column as the heading direction (cos, sin) formed in fp64 (TrajectoryController feeds row[9] to the yaw controller, main.py:58,
// and a direction makes psi and psi + 2 pi k the same set-point, as wrap_to_pi(wrap_to_2pi(psi_des) - psi) does, controller.py:156-168).
__global__ void __launch_bounds__(128) table_targets_kernel(const double* __restrict__ tables, long long n_rows, TargetRow* __restrict__ out) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_rows) return;
  const double* r = tables + g * 11;
  TargetRow t;
  t.x = r[0]; t.y = r[1]; t.z = r[2];
  t.vx = (float)r[3]; t.vy = (float)r[4]; t.vz = (float)r[5];
  t.ax = (float)r[6]; t.ay = (float)r[7]; t.az = (float)r[8];
  const double yaw = r[9];
  t.yc = (float)cos(yaw); t.ys = (float)sin(yaw);
  out[g] = t;
}

}  // namespace uavb

extern "C" int uavb_table_targets_f64(const double* tables, long long n_rows, void* targets_out, void* stream) {
  using namespace uavb;
  UAVB_REQUIRE(tables && targets_out, "table_targets: NULL pointer");
  UAVB_REQUIRE(n_rows >= 0, "table_targets: n_rows must be >= 0");
  int rc = require_device();
  if (rc) return rc;
  if (n_rows == 0) return UAVB_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long blocks = (n_rows + 127) / 128;
  UAVB_REQUIRE(blocks <= 0x7fffffffLL, "table_targets: too many rows");
  table_targets_kernel<<<(unsigned)blocks, 128, 0, st>>>(tables, n_rows, static_cast<TargetRow*>(targets_out));
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

extern "C" int uavb_rollout_tables_f32(const uavb_rollout_args* args, const uavb_table_set* tables, void* stream) {
  using namespace uavb;
  int rc = check_args(args, false, true);
  if (rc) return rc;
  UAVB_REQUIRE(tables != nullptr && tables->rows != nullptr, "rollout_tables: tables and tables->rows are required");
  UAVB_REQUIRE(tables->shared_rows >= 0, "rollout_tables: shared_rows must be >= 0");
  if (tables->shared_rows > 0) {
    UAVB_REQUIRE(tables->offsets == nullptr && tables->table_index == nullptr,
                 "rollout_tables: a shared table (shared_rows > 0) takes no offsets and no table_index");
  } else {
    UAVB_REQUIRE(tables->n_tables >= 1 && tables->offsets != nullptr, "rollout_tables: per-rollout tables need n_tables >= 1 and offsets");
    UAVB_REQUIRE(tables->table_index != nullptr || tables->n_tables == args->B || args->B == 0,
                 "rollout_tables: without table_index rollout b flies table b (n_tables == B)");
  }
  uavb_rollout_args a = *args;
  a.dt_outer = a.veh.dt * a.inner_per_outer;               // CascadedController.dt of the table's outer period (main.py:97)
  if (tables->shared_rows > 0) {                           // the shared-mission table kernels, unchanged
    a.shared_targets = tables->rows;
    a.n_target_rows = tables->shared_rows;
    return launch_rollout<float>(&a, stream, nullptr, true);
  }
  const TableSetDev ts{static_cast<const TargetRow*>(tables->rows), tables->offsets, tables->table_index};
  return launch_rollout<float>(&a, stream, &ts, true);
}

extern "C" int uavb_rollout_targets_f64(const double* seg_coeffs, const int* seg_rows, const int* seg_table, const double* seg_yaw0, int n_seg,
                                        double dt_outer, void* targets_out, int n_rows, void* stream) {
  using namespace uavb;
  static_assert(sizeof(TargetRow) == UAVB_TARGET_ROW_BYTES, "TargetRow layout");
  UAVB_REQUIRE(seg_coeffs && seg_rows && seg_table && seg_yaw0 && targets_out, "rollout_targets: NULL pointer");
  UAVB_REQUIRE(n_seg >= 1 && n_seg <= 255 && n_rows >= 0 && dt_outer > 0.0, "rollout_targets: 1 <= n_seg <= 255, n_rows >= 0, dt_outer > 0 required");
  int rc = require_device();
  if (rc) return rc;
  if (n_rows == 0) return UAVB_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  StreamScratch tmp(st);
  if (tmp.alloc((size_t)n_rows * (sizeof(float2) + sizeof(int))) != cudaSuccess) {
    cudaGetLastError();
    return set_error(UAVB_ENOMEM, "rollout_targets: scratch allocation failed");
  }
  float2* raw = static_cast<float2*>(tmp.p);
  int* tstart = reinterpret_cast<int*>(raw + n_rows);
  TargetRow* out = static_cast<TargetRow*>(targets_out);
  target_rows_kernel<<<div_up(n_rows, 128), 128, 0, st>>>(seg_coeffs, seg_rows, seg_table, n_seg, dt_outer, out, raw, tstart, n_rows);
  UAVB_CUDA_OK(cudaGetLastError());
  target_heading_kernel<<<div_up(n_rows, 128), 128, 0, st>>>(raw, tstart, seg_yaw0, seg_rows, n_seg, out, n_rows);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

// Development entry point, not part of uavb.h (tests/test_speculative_gpu.py, tools/spec_probe.py): force_exact = 1 flies every
// stretch of the speculative kernels with the exact body in later launches, 0 restores speculation.
extern "C" int uavb_dev_speculation(int force_exact) {
  uavb::g_spec_exact = force_exact != 0;
  return UAVB_OK;
}

extern "C" int uavb_rollout_f32(const uavb_rollout_args* args, void* stream) { return uavb::launch_rollout<float>(args, stream); }
extern "C" int uavb_rollout_f64(const uavb_rollout_args* args, void* stream) { return uavb::launch_rollout<double>(args, stream); }
extern "C" void uavb_vehicle_defaults(uavb_vehicle* veh) {
  if (veh) uavb::vehicle_defaults(veh);
}
