// rollout_pair.cuh -- the fp32 production rollout, two drones per thread: thread j of the launch flies drones 2j and
// 2j+1 in the two lanes of float2 registers (flight_pair.cuh: the 1 kHz tick in packed fp32x2 instructions); the 100 Hz
// outer loop is its packed restatement (outer_update_pair); the table cursor, the fp64 set-point evaluation and fold, and
// the collision flag are the scalar code of rollout_core.cuh run once per lane.  Both drones of a pair tick in lock-step (same tick count, same outer/inner schedule, main.py:37-45), so the
// schedule below is rollout_run's with every per-drone step done twice.
//
// A pair's two rollouts never mix: each lane runs exactly the operation sequence a lone drone would, so per-rollout
// results do not depend on the partner, on the batch size or on how a job is sharded (tests/test_rollout_gpu.py).
#pragma once

#include "flight_pair.cuh"
#include "rollout_core.cuh"
#include "tma.cuh"

#include <type_traits>

namespace uavb {

// Ticks per loop iteration of the unrolled bodies (rollout_run_pair): 2 beats 1 by 2 % on the headline launch and by 1-2 % with
// per-rollout tables (DESIGN.md), and beats 5 / 10 in the speculative loop (profiles/r03_spec_probe.jsonl: 4.40 against 4.43 / 4.54 ms).
constexpr int kTickUnroll = 2;

// [sample][13][B] state log of a pair: drones 2j, 2j+1 are neighbours in every field row, so a field leaves as ONE 8-byte
// streaming store per thread when the rows are 8-byte aligned (B even) -- a warp writes 256 contiguous bytes per field.
// `out` points at element 2j of field 0 of the next sample.
struct PairLog {
  static constexpr bool kNormEveryTick = true;
  float* out;
  unsigned B;              // field stride in elements
  int stride, left;
  bool vec, second;        // 8-byte stores possible; the pair's second drone exists
  UAVB_DEV void put(float* o, V2 x) const {
    if (vec) { __stcs(reinterpret_cast<float2*>(o), x); return; }
    __stcs(o, x.x);
    if (second) __stcs(o + 1, x.y);
  }
  UAVB_DEV void tick(const Drone2& d) {
    if (--left) return;
    left = stride;
    float* o = out;
    const unsigned b = B;
    put(o, make_float2((float)(d.px[0] + (double)d.dx.x), (float)(d.px[1] + (double)d.dx.y)));
    put(o + (size_t)b, make_float2((float)(d.py[0] + (double)d.dy.x), (float)(d.py[1] + (double)d.dy.y)));
    put(o + (size_t)(2u * b), make_float2((float)(d.pz[0] + (double)d.dz.x), (float)(d.pz[1] + (double)d.dz.y)));
    put(o + (size_t)(3u * b), d.q0); put(o + (size_t)(4u * b), d.q1); put(o + (size_t)(5u * b), d.q2); put(o + (size_t)(6u * b), d.q3);
    put(o + (size_t)(7u * b), d.vx); put(o + (size_t)(8u * b), d.vy); put(o + (size_t)(9u * b), d.vz);
    put(o + (size_t)(10u * b), d.wx); put(o + (size_t)(11u * b), d.wy); put(o + (size_t)(12u * b), d.wz);
    out = o + (size_t)(13u * b);
  }
};

// The same log through the TMA unit: every warp stages kLogTmaSamples samples x 13 fields x 64 drones in shared memory (one
// conflict-free 8-byte shared store per field and thread, 32-bit addressing) and its first lane sends the 13 kLogTmaSamples x 256-byte
// box to the [samples x 13][B] log with ONE tensor store -- instead of 13 global stores with 64-bit address arithmetic per thread
// and sample -- while the warp flies on into the second staging buffer.  Samples left over at the end of a slice leave through
// the one-sample map.  Drones past the end of the batch are clipped by the map (B is a multiple of 4 on this path).
constexpr int kLogTmaSamples = 2;
constexpr int kLogTmaSampleFloats = 13 * 64;               // one sample of one warp
constexpr int kLogTmaWarpFloats = 2 * kLogTmaSamples * kLogTmaSampleFloats;    // two buffers
struct alignas(64) LogTma {
  CUtensorMap box_k;       // boxes of (13 kLogTmaSamples) rows x 64 drones
  CUtensorMap box_1;       // boxes of 13 rows x 64 drones
  int stage_offset;        // byte offset of the staging area in dynamic shared memory (128-byte aligned)
};
struct PairLogTma {
  static constexpr bool kNormEveryTick = true;
  const LogTma* maps;
  float* stage;            // this warp's staging area
  float2* mine;            // ... + this lane's column pair in buffer 0, sample 0
  unsigned mask;           // lanes of the warp that fly (the others are past the end of the batch)
  int col, sample;         // tensor coordinates: first drone of the warp, index of the next sample to stage
  int stride, left, filled, buf;
  UAVB_DEV bool leader() const { return (threadIdx.x & 31u) == (unsigned)(__ffs(mask) - 1); }
  UAVB_DEV void send(const CUtensorMap* map, const float* src, int first_sample) {
    fence_proxy_async_smem();                              // every lane: its staged columns before the async-proxy read
    __syncwarp(mask);
    if (leader()) {
      tensor_store_2d(map, col, first_sample * 13, src);
      bulk_commit();
      bulk_wait_read<1>();                                 // the OTHER buffer's store has finished reading: it may be refilled
    }
    __syncwarp(mask);
  }
  UAVB_DEV void tick(const Drone2& d) {
    if (--left) return;
    left = stride;
    float2* o = mine + (buf * kLogTmaSamples + filled) * (kLogTmaSampleFloats / 2);
    o[0 * 32] = make_float2((float)(d.px[0] + (double)d.dx.x), (float)(d.px[1] + (double)d.dx.y));
    o[1 * 32] = make_float2((float)(d.py[0] + (double)d.dy.x), (float)(d.py[1] + (double)d.dy.y));
    o[2 * 32] = make_float2((float)(d.pz[0] + (double)d.dz.x), (float)(d.pz[1] + (double)d.dz.y));
    o[3 * 32] = d.q0; o[4 * 32] = d.q1; o[5 * 32] = d.q2; o[6 * 32] = d.q3;
    o[7 * 32] = d.vx; o[8 * 32] = d.vy; o[9 * 32] = d.vz;
    o[10 * 32] = d.wx; o[11 * 32] = d.wy; o[12 * 32] = d.wz;
    ++sample;
    if (++filled == kLogTmaSamples) {
      send(&maps->box_k, stage + buf * kLogTmaSamples * kLogTmaSampleFloats, sample - kLogTmaSamples);
      buf ^= 1; filled = 0;
    }
  }
  // end of the slice: the samples still staged, one box each; then the staging area is free for the CTA's next work item
  UAVB_DEV void finish() {
    for (int k = 0; k < filled; ++k) send(&maps->box_1, stage + (buf * kLogTmaSamples + k) * kLogTmaSampleFloats, sample - filled + k);
    filled = 0;
    if (leader()) bulk_wait_read<0>();
    __syncwarp(mask);
  }
};

// D5, the viewer's flown-path list (MujocoSimulation._record_actual_trajectory, mujoco_sim.py:201-218) for the pair: `time` is
// data.time -- mj_step adds the time step once per tick, so it is accumulated the same way, one fp64 addition per tick, and the
// sample ticks come out as the reference's (50 or 51 ticks apart at 20 Hz) -- the gate is quad.z > takeoff z => skip, the
// sample time rule time < next => skip, next = time + interval.  Positions are stored as fp32 triples [sample][3][B].
// Quaternion handling is the metrics-only one (kNormEveryTick = false): a rollout that records its path flies the metrics-only
// rollout to a few ulps (another compiled kernel; measured 2e-7 after 10 760 ticks).
struct PairTrajLog {
  static constexpr bool kNormEveryTick = false;
  float* out;              // element (sample 0, field 0, drone 2j)
  long long B;
  double time, dt, interval, gate_z;
  double next[2];
  int count[2];
  int max_samples;
  bool second;             // the pair's second drone exists
  template <int L> UAVB_DEV void lane_tick(const Drone2& d) {
    const double z = d.pz[L] + (double)lane<L>(d.dz);
    if (z > gate_z || time < next[L]) return;             // comparisons with NaN are false, as in the reference's two tests
    if (count[L] < max_samples && (L == 0 || second)) {
      float* o = out + (size_t)count[L] * 3 * B + L;
      o[0] = (float)(d.px[L] + (double)lane<L>(d.dx)); o[B] = (float)(d.py[L] + (double)lane<L>(d.dy)); o[2 * B] = (float)z;
    }
    ++count[L];
    next[L] = time + interval;
  }
  UAVB_DEV void tick(const Drone2& d) {
    time += dt;
    lane_tick<0>(d);
    lane_tick<1>(d);
  }
};

struct NoPairLog {
  static constexpr bool kNormEveryTick = false;
  UAVB_DEV void tick(const Drone2&) {}
};

// Where a pair's set-points come from (a compile-time switch of the kernel, so each body carries only its own code):
//   kTargetFly         each lane evaluates its own mission's splines in fp64 (MissionView cursor);
//   kTargetShared      one precomputed TargetRow table for every rollout (MissionView::trows), one row serves both lanes;
//   kTargetPerRollout  each lane reads its own precomputed table (MissionView::trows / n_trows of the lane), e.g. caller-supplied
//                      (N, 11) trajectory tables converted by uavb_table_targets_f64.
enum : int { kTargetFly = 0, kTargetShared = 1, kTargetPerRollout = 2 };

// Speculative stretches (metrics-only bodies of the shared-table and per-rollout-table modes).  The exact tick carries two rare
// paths -- the rotor-limit path and the large-rotation quaternion map -- and the branch around each keeps the next tick's head
// from being scheduled against this tick's body.  A non-watching stretch therefore flies the branch-free inner_tick_pair_spec, with
// the fields the tick writes checkpointed in shared memory first; when some lane of the warp would have taken a rare path, the warp
// reloads the checkpoint and flies the same ticks with the exact body.  Without a rare path both bodies execute the same rounded
// operations, so results are bit-identical either way.  Measured in DESIGN.md (K2, speculative stretches).
// Non-watching stretches flown with the exact body after a rollback (rare paths cluster in mission phases): 4 against 0 / 16 gives
// 4.40 against 4.64 / 4.41 ms (profiles/r03_spec_probe.jsonl).
constexpr int kSpecHold = 4;

// The tan-form quaternion map of the pair tick grows |q| by 1/cos(dt |w| / 2) per tick on purpose, and renormalise_q_pair's
// 1.5 - 0.5 |q|^2 is exact to O(e^2) only: the metrics-only bodies renormalise at every phase that is a multiple of kNormTicks as well as
// at the end of each outer period, so that periods longer than 10 ticks (frequency > 10) let the norm grow no further than at 10.
constexpr int kNormTicks = 10;
constexpr int kSpecSlotVec4 = 10;                            // 20 float2 fields of Drone2 = 10 x 16 bytes per thread
template <int MODE, class LOG> constexpr bool kSpecBody = std::is_same<LOG, NoPairLog>::value && MODE != kTargetFly;

// One thread's checkpoint in dynamic shared memory: 16-byte words k = 0..9 at s_spec[base + 32 k], base = the slot area (after the
// staged boxes) + 320 words per warp + the lane -- a warp's store of one word is 512 contiguous bytes, conflict-free, and the
// addresses are 32-bit shared-window offsets.
extern __shared__ __align__(16) float4 s_spec[];
struct SpecSlot {
  int base;
  int exact;               // development switch (uavb_dev_speculation): fly every stretch with the exact body
  UAVB_DEV float4& w(int k) const { return s_spec[base + 32 * k]; }
  UAVB_DEV void save(const Drone2& d) const {
    w(0) = make_float4(d.dx.x, d.dx.y, d.dy.x, d.dy.y);
    w(1) = make_float4(d.dz.x, d.dz.y, d.q0.x, d.q0.y);
    w(2) = make_float4(d.q1.x, d.q1.y, d.q2.x, d.q2.y);
    w(3) = make_float4(d.q3.x, d.q3.y, d.vx.x, d.vx.y);
    w(4) = make_float4(d.vy.x, d.vy.y, d.vz.x, d.vz.y);
    w(5) = make_float4(d.wx.x, d.wx.y, d.wy.x, d.wy.y);
    w(6) = make_float4(d.wz.x, d.wz.y, d.om0.x, d.om0.y);
    w(7) = make_float4(d.om1.x, d.om1.y, d.om2.x, d.om2.y);
    w(8) = make_float4(d.om3.x, d.om3.y, d.zbx.x, d.zbx.y);
    w(9) = make_float4(d.zby.x, d.zby.y, d.zbz.x, d.zbz.y);
  }
  UAVB_DEV void load(Drone2& d) const {
    float4 t;
    t = w(0); d.dx = make_float2(t.x, t.y); d.dy = make_float2(t.z, t.w);
    t = w(1); d.dz = make_float2(t.x, t.y); d.q0 = make_float2(t.z, t.w);
    t = w(2); d.q1 = make_float2(t.x, t.y); d.q2 = make_float2(t.z, t.w);
    t = w(3); d.q3 = make_float2(t.x, t.y); d.vx = make_float2(t.z, t.w);
    t = w(4); d.vy = make_float2(t.x, t.y); d.vz = make_float2(t.z, t.w);
    t = w(5); d.wx = make_float2(t.x, t.y); d.wy = make_float2(t.z, t.w);
    t = w(6); d.wz = make_float2(t.x, t.y); d.om0 = make_float2(t.z, t.w);
    t = w(7); d.om1 = make_float2(t.x, t.y); d.om2 = make_float2(t.z, t.w);
    t = w(8); d.om3 = make_float2(t.x, t.y); d.zbx = make_float2(t.z, t.w);
    t = w(9); d.zby = make_float2(t.x, t.y); d.zbz = make_float2(t.z, t.w);
  }
};

// Set-points of the coming outer period and the position errors (set-point - position, fp64, rounded once): one table row
// for both lanes of a shared mission, otherwise each lane's own cursor or table.
template <int MODE> struct PairTarget;
template <> struct PairTarget<kTargetShared> {
  typedef float T;
  static UAVB_DEV void fetch(const Drone2& d, Cursor<float> (&c)[2], const MissionView& ma, const MissionView&, Target2<float>& t2, V2& ex, V2& ey, V2& ez) {
    Target<float> t;
    table_target<float>(ma.trows, c[0].row, &t);
    if (c[0].row + 1 < ma.n_trows) ++c[0].row;               // index clamp of main.py:61
    c[1].row = c[0].row;
    // the row of the NEXT outer period, one stretch of ticks ahead: into L1 now, so that its loads do not wait on L2 then
    const char* nxt = reinterpret_cast<const char*>(ma.trows + c[0].row);
    asm volatile("prefetch.global.L1 [%0];" ::"l"(nxt));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(nxt + sizeof(TargetRow) - 4));
    t2.vx = t.vx; t2.vy = t.vy; t2.vz = t.vz; t2.ax = t.ax; t2.ay = t.ay; t2.az = t.az; t2.yc = t.yc; t2.ys = t.ys;
    ex = make_float2((float)(t.x - d.px[0]), (float)(t.x - d.px[1]));
    ey = make_float2((float)(t.y - d.py[0]), (float)(t.y - d.py[1]));
    ez = make_float2((float)(t.z - d.pz[0]), (float)(t.z - d.pz[1]));
  }
};
// Zip the set-points of the two lanes and form their position errors.
UAVB_DEV void zip_targets(const Drone2& d, const Target<float>& ta, const Target<float>& tb, Target2<V2>& t2, V2& ex, V2& ey, V2& ez) {
  t2.vx = make_float2(ta.vx, tb.vx); t2.vy = make_float2(ta.vy, tb.vy); t2.vz = make_float2(ta.vz, tb.vz);
  t2.ax = make_float2(ta.ax, tb.ax); t2.ay = make_float2(ta.ay, tb.ay); t2.az = make_float2(ta.az, tb.az);
  t2.yc = make_float2(ta.yc, tb.yc); t2.ys = make_float2(ta.ys, tb.ys);
  ex = make_float2((float)(ta.x - d.px[0]), (float)(tb.x - d.px[1]));
  ey = make_float2((float)(ta.y - d.py[0]), (float)(tb.y - d.py[1]));
  ez = make_float2((float)(ta.z - d.pz[0]), (float)(tb.z - d.pz[1]));
}
template <> struct PairTarget<kTargetFly> {
  typedef V2 T;
  static UAVB_DEV void fetch(const Drone2& d, Cursor<float> (&c)[2], const MissionView& ma, const MissionView& mb, Target2<V2>& t2, V2& ex, V2& ey, V2& ez) {
    Target<float> ta, tb;
    cursor_target<float>(c[0], ma, &ta);
    cursor_advance(&c[0].seg, &c[0].row, ma);
    cursor_target<float>(c[1], mb, &tb);
    cursor_advance(&c[1].seg, &c[1].row, mb);
    zip_targets(d, ta, tb, t2, ex, ey, ez);
  }
};
template <> struct PairTarget<kTargetPerRollout> {
  typedef V2 T;
  static UAVB_DEV void fetch(const Drone2& d, Cursor<float> (&c)[2], const MissionView& ma, const MissionView& mb, Target2<V2>& t2, V2& ex, V2& ey, V2& ez) {
    Target<float> ta, tb;
    table_target<float>(ma.trows, c[0].row, &ta);
    if (c[0].row + 1 < ma.n_trows) ++c[0].row;               // index clamp of main.py:61, with the lane's own row count
    table_target<float>(mb.trows, c[1].row, &tb);
    if (c[1].row + 1 < mb.n_trows) ++c[1].row;
    // each lane's row of the NEXT outer period into L1, as for the shared table: 5 % once the tables leave L2 (DESIGN.md)
    const char* na = reinterpret_cast<const char*>(ma.trows + c[0].row);
    const char* nb = reinterpret_cast<const char*>(mb.trows + c[1].row);
    asm volatile("prefetch.global.L1 [%0];" ::"l"(na));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(na + sizeof(TargetRow) - 4));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(nb));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(nb + sizeof(TargetRow) - 4));
    zip_targets(d, ta, tb, t2, ex, ey, ez);
  }
};

// Obstacle culling for the coming stretch of n ticks (rollout_run, "clearance budget"): true when either drone could reach a
// box before the next check, i.e. the per-tick inclusive test must run.  `clear` = lower bounds of the Chebyshev gaps.
// With a floor (Ground) the gap also counts the room above it, and a drone keeps being watched after its collision flag is set.
template <int L, class OBST> UAVB_DEV float pair_gap(const Drone2& d, const Accum<float>& a, const OBST& o, const Ground& gr) {
  const double z = d.pz[L] + (double)lane<L>(d.dz);
  float g = a.collided ? 3.0e38f : o.gap((float)(d.px[L] + (double)lane<L>(d.dx)), (float)(d.py[L] + (double)lane<L>(d.dy)), (float)z);
  if (gr.on) {
    const float gg = (float)(gr.z - z);
    g = (gg < g || gg != gg) ? gg : g;
  }
  return g;
}
template <class OBST> UAVB_DEV bool pair_watch(const Drone2& d, const Accum<float> (&a)[2], const VehU<float>& u, V2 acc_max,
                                               const OBST& oa, const OBST& ob, int n, V2& clear, const Ground& gr) {
  const float T = __fmul_rn((float)n, u.dt);
  const V2 speed = sqrt2(fma2(d.vx, d.vx, fma2(d.vy, d.vy, mul2(d.vz, d.vz))));
  const V2 reach = fma2(mul2(fma2(acc_max, T, speed), T), 1.01f, 1e-4f);
  const bool live_a = !a[0].collided || gr.on, live_b = !a[1].collided || gr.on;
  if ((live_a && !(clear.x > reach.x)) || (live_b && !(clear.y > reach.y))) {      // measure (rare): NaN positions keep measuring
    if (live_a && !(clear.x > reach.x)) clear.x = pair_gap<0>(d, a[0], oa, gr);
    if (live_b && !(clear.y > reach.y)) clear.y = pair_gap<1>(d, a[1], ob, gr);
  }
  const bool watch = (live_a && !(clear.x > reach.x)) || (live_b && !(clear.y > reach.y));
  clear = sub2(clear, reach);
  return watch;
}

// The floor for lane L after a tick: below it => back onto it, no downward velocity (NED: +z is down).
template <int L> UAVB_DEV void pair_floor(Drone2& d, const Ground& gr) {
  if (d.pz[L] + (double)lane<L>(d.dz) > gr.z) {
    lane<L>(d.dz) = (float)(gr.z - d.pz[L]);
    lane<L>(d.vz) = fminf(lane<L>(d.vz), 0.f);
  }
}

template <int L, class OBST> UAVB_DEV void pair_hit(const Drone2& d, Accum<float>& a, const OBST& obst, int tick) {
  if (!a.collided && obst.hit((float)(d.px[L] + (double)lane<L>(d.dx)), (float)(d.py[L] + (double)lane<L>(d.dy)), (float)(d.pz[L] + (double)lane<L>(d.dz)))) {
    a.collided = 1; a.first_hit = tick;
  }
}

// n_ticks ticks of the closed loop for the pair; the schedule, the obstacle culling and the metrics are rollout_run's
// (rollout_core.cuh), see there.  c[0].phase is the phase of both lanes.  VP2: VehP2 or VehP<float> (see inner_tick_pair).
// LAG (thrust_frame_lag of the launch) is a compile-time switch of the kernel: one stretch body per (kernel, watch) keeps the
// instruction footprint of a warp's working set inside the instruction cache (ncu: with all four (watch, lag) bodies in one kernel
// the per-rollout-mission workload spent as long waiting for instructions as for operands).
// MODE: kTargetFly / kTargetShared / kTargetPerRollout (PairTarget above).
template <int MODE, bool LAG, class VP2, class OBST, class LOG>
UAVB_DEV void rollout_run_pair(Drone2& d, Cursor<float> (&c)[2], Accum<float> (&a)[2], const VehU<float>& u, const VehP<float>& va,
                               const VehP<float>& vb, const VP2& v2, const VehO2& vo, const MissionView& ma, const MissionView& mb, int tick0,
                               int n_ticks, int freq, const OBST& oa, const OBST& ob, LOG& logger, const Ground gr = Ground{0, 0.0},
                               const SpecSlot slot = SpecSlot{0, 0}) {
  int k = 0;
  V2 clear = make_float2(0.f, 0.f);                          // not part of the carry: every launch / slice measures first
  const V2 acc_max = make_float2(va.acc_max, vb.acc_max);
  constexpr bool kSpec = kSpecBody<MODE, LOG>;
  int hold = 0;                                              // non-watching stretches left to fly exactly (not carried: no effect on results)
  if constexpr (kSpec) hold = slot.exact ? 0x7fffffff : 0;
  // periods longer than kNormTicks split their stretches (below); a separate copy of the loop, so that shorter periods fly the same
  // code as without the split, and one tick per iteration there (unrolled, the second copy of the body spills at 255 registers).
  // kTargetFly bodies (fp64 set-points evaluated inline) keep one loop that splits at run time: a second copy spills there.
  const bool long_period = !LOG::kNormEveryTick && freq > kNormTicks;   // (launch-uniform)
  auto run = [&](auto long_c) {
  constexpr bool kLong = decltype(long_c)::value;
  while (k < n_ticks) {
    if (c[0].phase == 0) {
      Target2<typename PairTarget<MODE>::T> t;
      V2 ex, ey, ez;
      PairTarget<MODE>::fetch(d, c, ma, mb, t, ex, ey, ez);    // the position is folded here (d.dx = 0)
      c[0].ex = ex.x; c[1].ex = ex.y; c[0].ey = ey.x; c[1].ey = ey.y; c[0].ez = ez.x; c[1].ez = ez.y;
      outer_update_pair(d, u, vo, t, ex, ey, ez);
    }
    // stretches also end where the phase reaches a multiple of kNormTicks (below): F <= kNormTicks keeps one stretch per period
    int n = (freq - c[0].phase < n_ticks - k) ? (freq - c[0].phase) : (n_ticks - k);
    if (kLong && long_period) {
      const int to_norm = kNormTicks - c[0].phase % kNormTicks;
      n = to_norm < n ? to_norm : n;
    }
    bool watch = false;
    if (OBST::kAny) watch = __any_sync(__activemask(), pair_watch(d, a, u, acc_max, oa, ob, n, clear, gr));   // one decision per warp; watching is always correct
    auto stretch = [&](auto watch_c) {
      constexpr bool kWatch = decltype(watch_c)::value;
      // two ticks per iteration (the tail of one tick overlaps the head of the next: +2 % on the table-driven headline workload)
      // only where the instruction footprint allows it: the watching bodies carry the per-tick box tests, and kernels that
      // evaluate the set-points on the fly carry two inlined fp64 evaluations per period -- unrolled, BASELINE configs[3]
      // waits for instruction fetches and runs 10 % slower (measured).  Per-rollout tables unroll only without a state log: with
      // Monte-Carlo overrides and per-thread log stores the unrolled body no longer fits 255 registers (ptxas spills), and a
      // logging launch is bound by its HBM stores anyway.
#pragma unroll((kLong || kWatch || MODE == kTargetFly || (MODE == kTargetPerRollout && LOG::kNormEveryTick)) ? 1 : kTickUnroll)
      for (int j = 0; j < n; ++j) {
        inner_tick_pair<LOG::kNormEveryTick, LAG>(d, u, v2);
        if constexpr (kWatch) {
          if (gr.on) { pair_floor<0>(d, gr); pair_floor<1>(d, gr); }
          pair_hit<0>(d, a[0], oa, tick0 + k + j);
          pair_hit<1>(d, a[1], ob, tick0 + k + j);
        }
        logger.tick(d);
      }
    };
    if constexpr (kSpec) {
      bool flown = false;
      if (!watch && hold == 0) {                             // (warp-uniform)
        slot.save(d);
        unsigned rare = 0;
#pragma unroll(!kLong && (LAG || !std::is_same<VP2, VehP2>::value) ? kTickUnroll : 1)
        for (int j = 0; j < n; ++j) inner_tick_pair_spec<LAG>(d, u, v2, rare);
        flown = !__any_sync(__activemask(), rare != 0);
        if (!flown) {                                        // roll back: the same n ticks with the exact body
          slot.load(d);
          hold = kSpecHold + 1;
        }
      }
      if (!watch && hold > 0) --hold;
      if (watch) {
        stretch(BoolC<true>{});
      } else if (!flown) {
        stretch(BoolC<false>{});
      }
    } else {
      if (watch) {
        stretch(BoolC<true>{});
      } else {
        stretch(BoolC<false>{});
      }
    }
    k += n;
    c[0].phase += n;
    if (c[0].phase == freq) {
      c[0].phase = 0;
      if (!LOG::kNormEveryTick) renormalise_q_pair(d);       // once per outer period (not per launch: chunked runs stay bit-identical)
      // tracking error |set-point - p| after the period (test_mujoco_trajectory_tracking.py:27-31): p = fold + displacement
      const V2 fx = sub2(make_float2(c[0].ex, c[1].ex), d.dx), fy = sub2(make_float2(c[0].ey, c[1].ey), d.dy), fz = sub2(make_float2(c[0].ez, c[1].ez), d.dz);
      const V2 e2 = fma2(fx, fx, fma2(fy, fy, mul2(fz, fz)));
      const V2 e = sqrt2(e2);
      const V2 se = add2(make_float2(a[0].sum_e, a[1].sum_e), e), se2 = add2(make_float2(a[0].sum_e2, a[1].sum_e2), e2);
      a[0].sum_e = se.x; a[1].sum_e = se.y; a[0].sum_e2 = se2.x; a[1].sum_e2 = se2.y;
      a[0].max_e = fmaxf(a[0].max_e, e.x); a[1].max_e = fmaxf(a[1].max_e, e.y);
      ++a[0].periods; ++a[1].periods;
      // fold the displacement into the fp64 position
      d.px[0] += (double)d.dx.x; d.py[0] += (double)d.dy.x; d.pz[0] += (double)d.dz.x;
      d.px[1] += (double)d.dx.y; d.py[1] += (double)d.dy.y; d.pz[1] += (double)d.dz.y;
      d.dx = d.dy = d.dz = make_float2(0.f, 0.f);
    } else if (kLong && long_period && c[0].phase % kNormTicks == 0) {
      renormalise_q_pair(d);   // within a long period too, on the phase (not where a launch ends)
    }
    c[1].phase = c[0].phase;
  }
  };
  if constexpr (MODE == kTargetFly) {
    run(BoolC<!LOG::kNormEveryTick>{});
  } else {
    if (long_period) run(BoolC<true>{}); else run(BoolC<false>{});
  }
#pragma unroll
  for (int l = 0; l < 2; ++l) {
    if (!Math<float>::finite(a[l].sum_e2)) a[l].status |= 1;
    if (a[l].max_e > 1e4f) a[l].status |= 2;                 // more than 1e4 m from its set-point
  }
}

}  // namespace uavb
