// flight_pair.cuh -- the 1 kHz tick of the fp32 production rollout for TWO drones per thread, every state variable a float2
// (lane x = first drone, lane y = second drone), written with the packed fp32x2 instructions of sm_100
// (FFMA2 / FADD2 / FMUL2: fma.rn.f32x2, add.rn.f32x2, mul.rn.f32x2).
//
// Why two drones per thread (measured, profiles/r02_ffma2_probe.md): a packed instruction occupies the FMA pipe for two
// cycles but only ONE issue slot, and it has no lane swizzle -- both lanes must be the same operation on aligned register
// pairs.  The tick of one drone is full of horizontal products (cross products, the quaternion product, the mixer and the
// rotor-sum butterflies), so packing inside one drone costs as many moves as it saves; across two drones every operation
// of the tick is vertical.  The scalar tick was issue-bound (148 issue slots per drone-tick, FMA pipe 61 % busy); the pair
// tick is FMA-pipe-bound.
//
// Same equations, same order, same reference lines as inner_tick<float> in flight_core.cuh (controller.py:115-130,
// quad.py:88-122, mujoco_sim.py:232-255 + the restated free-body step) in the same "rotor units".  Every operation is an
// explicit IEEE round-to-nearest intrinsic (no compiler contraction), so a drone's trajectory does not depend on which
// lane it sits in, on its partner, or on the template instantiation that flies it.
//
// The 100 Hz outer loop (outer_update_pair) is the packed restatement of outer_update<float>: same stages, same order,
// explicit operations; MUFU functions, min / max / select run per lane.  Device-only.
#pragma once

#include "flight_core.cuh"

namespace uavb {

typedef float2 V2;

#define UAVB_DEV __device__ __forceinline__

UAVB_DEV V2 as2(V2 x) { return x; }
UAVB_DEV V2 as2(float x) { return make_float2(x, x); }            // becomes a 32-bit operand broadcast to both lanes (R.F32 / UR.F32)
UAVB_DEV V2 neg2(V2 x) { return make_float2(-x.x, -x.y); }        // folds into the operand's negate modifier
UAVB_DEV float neg2(float x) { return -x; }
UAVB_DEV V2 abs2(V2 x) { return make_float2(fabsf(x.x), fabsf(x.y)); }   // folds into the |abs| modifier
template <class A, class B, class C> UAVB_DEV V2 fma2(A a, B b, C c) { return __ffma2_rn(as2(a), as2(b), as2(c)); }
template <class A, class B> UAVB_DEV V2 add2(A a, B b) { return __fadd2_rn(as2(a), as2(b)); }
template <class A, class B> UAVB_DEV V2 sub2(A a, B b) { return __fadd2_rn(as2(a), neg2(as2(b))); }
template <class A, class B> UAVB_DEV V2 mul2(A a, B b) { return __fmul2_rn(as2(a), as2(b)); }
UAVB_DEV V2 clamp_pair(V2 x, float lo, float hi) { return make_float2(fminf(fmaxf(x.x, lo), hi), fminf(fmaxf(x.y, lo), hi)); }
UAVB_DEV V2 sqrt2(V2 x) { return make_float2(Math<float>::sqrt_fast(x.x), Math<float>::sqrt_fast(x.y)); }
template <int L> UAVB_DEV float& lane(V2& v) { return L ? v.y : v.x; }
template <int L> UAVB_DEV float lane(const V2& v) { return L ? v.y : v.x; }

// Per-rollout constants of the 1 kHz body for a pair with Monte-Carlo overrides (lane = drone).  Without overrides the
// tick reads the scalar VehP<float> of the kernel parameter block instead and every constant is a broadcast operand.
struct VehP2 {
  V2 kf_dt_over_m2, Gx, Gy, Gz, Jp, Jq, Jr, Wx, Wy, Wz, Kx, Ky, Kz, dvx, dvy, dvz;
};
UAVB_DEV void zip_vehp(VehP2& o, const VehP<float>& a, const VehP<float>& b) {
  o.kf_dt_over_m2 = make_float2(a.kf_dt_over_m2, b.kf_dt_over_m2);
  o.Gx = make_float2(a.Gx, b.Gx); o.Gy = make_float2(a.Gy, b.Gy); o.Gz = make_float2(a.Gz, b.Gz);
  o.Jp = make_float2(a.Jp, b.Jp); o.Jq = make_float2(a.Jq, b.Jq); o.Jr = make_float2(a.Jr, b.Jr);
  o.Wx = make_float2(a.Wx, b.Wx); o.Wy = make_float2(a.Wy, b.Wy); o.Wz = make_float2(a.Wz, b.Wz);
  o.Kx = make_float2(a.Kx, b.Kx); o.Ky = make_float2(a.Ky, b.Ky); o.Kz = make_float2(a.Kz, b.Kz);
  o.dvx = make_float2(a.dvx, b.dvx); o.dvy = make_float2(a.dvy, b.dvy); o.dvz = make_float2(a.dvz, b.dvz);
}

// Persistent state of the pair (registers across a whole slice).  Fields as in Drone<float>; the fp64 fold position and
// the 100 Hz scalars are kept per lane.
struct Drone2 {
  double px[2], py[2], pz[2];
  V2 dx, dy, dz;
  V2 q0, q1, q2, q3;
  V2 vx, vy, vz;
  V2 wx, wy, wz;
  V2 om0, om1, om2, om3;
  V2 coll, cp, cq, cr;
  V2 margin;           // rotor-limit margin of the current collective share (set_margin), refreshed with coll
  V2 zbx, zby, zbz;
  float integral[2], thrust_cmd[2];
};

// Room of the collective share `coll` inside the rotor limits (rotor units), shrunk by a few ulps of the upper limit: while
// |p_bar| + |q_bar| + |r_bar| stays below it, every mixer output coll +- r_bar +- p_bar +- q_bar lies inside [lo, hi] whatever the
// rounding of its three additions, i.e. the exact test of mix_and_limit passes.  The tick uses it as a cheap SUFFICIENT test; when it
// fails the exact path runs, so results never depend on it.
UAVB_DEV float limit_margin(float coll, float lo, float hi) { return fminf(coll - lo, hi - coll) - 1e-6f * hi; }

template <int L> UAVB_DEV void get_lane(const Drone2& p, Drone<float>& d) {
  d.px = p.px[L]; d.py = p.py[L]; d.pz = p.pz[L];
  d.dx = lane<L>(p.dx); d.dy = lane<L>(p.dy); d.dz = lane<L>(p.dz);
  d.q0 = lane<L>(p.q0); d.q1 = lane<L>(p.q1); d.q2 = lane<L>(p.q2); d.q3 = lane<L>(p.q3);
  d.vx = lane<L>(p.vx); d.vy = lane<L>(p.vy); d.vz = lane<L>(p.vz);
  d.wx = lane<L>(p.wx); d.wy = lane<L>(p.wy); d.wz = lane<L>(p.wz);
  d.om0 = lane<L>(p.om0); d.om1 = lane<L>(p.om1); d.om2 = lane<L>(p.om2); d.om3 = lane<L>(p.om3);
  d.integral = p.integral[L]; d.thrust_cmd = p.thrust_cmd[L]; d.coll = lane<L>(p.coll);
  d.pc = d.qc = d.rc = 0.f;                           // SI body-rate commands: not carried by the persistent rollout
  d.cp = lane<L>(p.cp); d.cq = lane<L>(p.cq); d.cr = lane<L>(p.cr);
  d.zbx = lane<L>(p.zbx); d.zby = lane<L>(p.zby); d.zbz = lane<L>(p.zbz);
}
template <int L> UAVB_DEV void put_lane(Drone2& p, const Drone<float>& d, const VehU<float>& u) {
  lane<L>(p.margin) = limit_margin(d.coll, u.w2min, u.w2max);
  p.px[L] = d.px; p.py[L] = d.py; p.pz[L] = d.pz;
  lane<L>(p.dx) = d.dx; lane<L>(p.dy) = d.dy; lane<L>(p.dz) = d.dz;
  lane<L>(p.q0) = d.q0; lane<L>(p.q1) = d.q1; lane<L>(p.q2) = d.q2; lane<L>(p.q3) = d.q3;
  lane<L>(p.vx) = d.vx; lane<L>(p.vy) = d.vy; lane<L>(p.vz) = d.vz;
  lane<L>(p.wx) = d.wx; lane<L>(p.wy) = d.wy; lane<L>(p.wz) = d.wz;
  lane<L>(p.om0) = d.om0; lane<L>(p.om1) = d.om1; lane<L>(p.om2) = d.om2; lane<L>(p.om3) = d.om3;
  p.integral[L] = d.integral; p.thrust_cmd[L] = d.thrust_cmd; lane<L>(p.coll) = d.coll;
  lane<L>(p.cp) = d.cp; lane<L>(p.cq) = d.cq; lane<L>(p.cr) = d.cr;
  lane<L>(p.zbx) = d.zbx; lane<L>(p.zby) = d.zby; lane<L>(p.zbz) = d.zbz;
}
// Mixer + rotor limits (quad.py:105-122) in rotor units for the pair.  The unclipped outputs come from the packed
// butterfly.  |p_bar| + |q_bar| + |r_bar| <= margin (see limit_margin) proves them inside the limits with three instructions.  A
// pair that fails it runs the limit path for BOTH lanes as straight-line packed code (a saturating lane must not cost its warp a
// chain of branch diamonds -- in BASELINE configs[3] some lane of a warp is at a limit in most ticks): the exact test of
// quad.py:114-121 per lane, the ratio scaling of :116-119 and the clip; a lane whose unclipped outputs pass the exact test keeps
// them.  Same operations as mix_and_limit<float> (flight_core.cuh), see there for the two-reciprocal form of the ratios.
UAVB_DEV float limit_scale(float m_hi, float m_lo, float room_hi, float room_lo) {
  const float l_hi = (m_hi > 0.f) ? __fmul_rn(room_hi, Math<float>::rcp_fast(m_hi)) : 1.f;
  const float l_lo = (m_lo < 0.f) ? __fmul_rn(room_lo, Math<float>::rcp_fast(m_lo)) : 1.f;
  return fminf(fmaxf(fminf(l_hi, l_lo), 0.f), 1.f);
}
UAVB_DEV void mix_and_limit_pair(V2 pb, V2 qb, V2 rb, V2 coll, V2 margin, float lo, float hi, V2& f0, V2& f1, V2& f2, V2& f3) {
  const V2 s1 = add2(pb, qb), s2 = sub2(pb, qb), t1 = add2(coll, rb), t2 = sub2(coll, rb);
  f0 = add2(t1, s1); f1 = sub2(t2, s2); f2 = sub2(t1, s1); f3 = add2(t2, s2);
  const V2 need = add2(add2(abs2(pb), abs2(qb)), abs2(rb));
  if (!(need.x <= margin.x && need.y <= margin.y)) {
    const bool ok_x = fmaxf(fmaxf(f0.x, f1.x), fmaxf(f2.x, f3.x)) <= hi && fminf(fminf(f0.x, f1.x), fminf(f2.x, f3.x)) >= lo;
    const bool ok_y = fmaxf(fmaxf(f0.y, f1.y), fmaxf(f2.y, f3.y)) <= hi && fminf(fminf(f0.y, f1.y), fminf(f2.y, f3.y)) >= lo;
    const V2 m0 = add2(s1, rb), m1 = neg2(add2(s2, rb)), m2 = sub2(rb, s1), m3 = sub2(s2, rb);
    const V2 room_hi = sub2(hi, coll), room_lo = sub2(lo, coll);          // >= 0 and <= 0: coll is a clipped collective share
    const V2 sc = make_float2(limit_scale(fmaxf(fmaxf(m0.x, m1.x), fmaxf(m2.x, m3.x)), fminf(fminf(m0.x, m1.x), fminf(m2.x, m3.x)), room_hi.x, room_lo.x),
                              limit_scale(fmaxf(fmaxf(m0.y, m1.y), fmaxf(m2.y, m3.y)), fminf(fminf(m0.y, m1.y), fminf(m2.y, m3.y)), room_hi.y, room_lo.y));
    const V2 g0 = clamp_pair(fma2(sc, m0, coll), lo, hi), g1 = clamp_pair(fma2(sc, m1, coll), lo, hi);
    const V2 g2 = clamp_pair(fma2(sc, m2, coll), lo, hi), g3 = clamp_pair(fma2(sc, m3, coll), lo, hi);
    f0 = make_float2(ok_x ? f0.x : g0.x, ok_y ? f0.y : g0.y); f1 = make_float2(ok_x ? f1.x : g1.x, ok_y ? f1.y : g1.y);
    f2 = make_float2(ok_x ? f2.x : g2.x, ok_y ? f2.y : g2.y); f3 = make_float2(ok_x ? f3.x : g3.x, ok_y ? f3.y : g3.y);
  }
}

// Asymmetric motor lag (quad.py:98-103): w += a_mean e + a_hdiff |e|, e = cmd - w.
UAVB_DEV void lag_toward_pair(Drone2& d, const VehU<float>& u, V2 c0, V2 c1, V2 c2, V2 c3) {
  const V2 e0 = sub2(c0, d.om0), e1 = sub2(c1, d.om1), e2 = sub2(c2, d.om2), e3 = sub2(c3, d.om3);
  d.om0 = fma2(u.a_hdiff, abs2(e0), fma2(u.a_mean, e0, d.om0));
  d.om1 = fma2(u.a_hdiff, abs2(e1), fma2(u.a_mean, e1, d.om1));
  d.om2 = fma2(u.a_hdiff, abs2(e2), fma2(u.a_mean, e2, d.om2));
  d.om3 = fma2(u.a_hdiff, abs2(e3), fma2(u.a_mean, e3, d.om3));
}

UAVB_DEV void renormalise_q_pair(Drone2& d) {
  const V2 nn = fma2(d.q0, d.q0, fma2(d.q1, d.q1, fma2(d.q2, d.q2, mul2(d.q3, d.q3))));
  const V2 rn = fma2(-0.5f, nn, 1.5f);
  d.q0 = mul2(d.q0, rn); d.q1 = mul2(d.q1, rn); d.q2 = mul2(d.q2, rn); d.q3 = mul2(d.q3, rn);
}

UAVB_DEV void half_axis_pair(const Drone2& d, V2& a, V2& b, V2& c) {
  a = fma2(d.q1, d.q3, mul2(d.q0, d.q2));
  b = fma2(d.q2, d.q3, neg2(mul2(d.q0, d.q1)));
  c = fma2(d.q1, d.q1, mul2(d.q2, d.q2));
}

// Quaternion map of the tick, q <- q * [cos(x), sin(x) w/|w|] with x = dt |w| / 2 (mju_quatIntegrate), in the form
//   n = q + q * (0, b),  b = (tan(x)/|w|) w        =>  n = q * [1, tan(x) w/|w|] = (q * [cos x, sin x w/|w|]) / cos x :
// the exact rotation with the norm grown by 1/cos(x) = 1 + x^2/2, which the renormalisation (once per outer period, or every
// tick under a state log) removes -- so neither cos(x) - 1 nor the four products q_i (cos(x) - 1) are formed per tick.
// tan(x)/x = 1 + x^2/3 + 2 x^4/15 ...: two terms are exact to half an ulp for x^2 < 5e-4 (|w| < 44.7 rad/s); a lane beyond
// that (a tumbling vehicle) takes the unit-norm sin / cos form with single-MUFU functions, as inner_tick<float> does.
UAVB_DEV void quat_step_large(float& q0, float& q1, float& q2, float& q3, float wx, float wy, float wz, float wn2, float h) {
  const float iw = Math<float>::rsqrt(wn2);
  float sn, cs;
  Math<float>::sincos_fast(__fmul_rn(h, __fmul_rn(wn2, iw)), &sn, &cs);
  const float sf = __fmul_rn(sn, iw), cm1 = __fadd_rn(cs, -1.f);
  const float bx = __fmul_rn(sf, wx), by = __fmul_rn(sf, wy), bz = __fmul_rn(sf, wz);
  const float n0 = __fadd_rn(q0, __fmaf_rn(-q3, bz, __fmaf_rn(-q2, by, __fmaf_rn(-q1, bx, __fmul_rn(q0, cm1)))));
  const float n1 = __fadd_rn(q1, __fmaf_rn(-q3, by, __fmaf_rn(q2, bz, __fmaf_rn(q0, bx, __fmul_rn(q1, cm1)))));
  const float n2 = __fadd_rn(q2, __fmaf_rn(q3, bx, __fmaf_rn(-q1, bz, __fmaf_rn(q0, by, __fmul_rn(q2, cm1)))));
  const float n3 = __fadd_rn(q3, __fmaf_rn(-q2, bx, __fmaf_rn(q1, by, __fmaf_rn(q0, bz, __fmul_rn(q3, cm1)))));
  q0 = n0; q1 = n1; q2 = n2; q3 = n3;
}

// One inner tick of the pair in the reference order; see inner_tick<float> for the derivation of the rotor-unit forms.
// VP: VehP2 (per-lane constants) or VehP<float> (launch-uniform constants, broadcast).  LAG: thrust along the body axis
// of the previous tick (stale data.xmat, SURVEY 3.2) or of this one.
template <bool NORM, bool LAG, class VP> UAVB_DEV void inner_tick_pair(Drone2& d, const VehU<float>& u, const VP& v) {
  const V2 yz = mul2(d.wy, d.wz), zx = mul2(d.wz, d.wx), xy = mul2(d.wx, d.wy);
  V2 w0, w1, w2, w3;
  mix_and_limit_pair(fma2(neg2(v.Jp), d.wx, fma2(v.Gx, yz, d.cp)), fma2(neg2(v.Jq), d.wy, fma2(v.Gy, zx, d.cq)),
                     fma2(neg2(v.Jr), d.wz, fma2(v.Gz, xy, d.cr)), d.coll, d.margin, u.w2min, u.w2max, w0, w1, w2, w3);
  lag_toward_pair(d, u, sqrt2(w0), sqrt2(w1), sqrt2(w2), sqrt2(w3));
  V2 ha, hb, hc;
  half_axis_pair(d, ha, hb, hc);
  const V2 ua = LAG ? d.zbx : ha, ub = LAG ? d.zby : hb, uc = LAG ? d.zbz : hc;
  d.zbx = ha; d.zby = hb; d.zbz = hc;
  // rotor sums (mujoco_sim.py:235-247): a = s0+s1, c = s0-s1, b = s2+s3, e = s2-s3 with s_i = w_i^2
  const V2 s0 = mul2(d.om0, d.om0), s2 = mul2(d.om2, d.om2);
  const V2 a = fma2(d.om1, d.om1, s0), c = fma2(neg2(d.om1), d.om1, s0);
  const V2 b = fma2(d.om3, d.om3, s2), e = fma2(neg2(d.om3), d.om3, s2);
  const V2 tot = add2(a, b), ty = sub2(a, b), tx = sub2(c, e), tzn = add2(c, e);
  const V2 dvt2 = mul2(neg2(tot), v.kf_dt_over_m2);
  // semi-implicit Euler: velocity increments formed first (thrust and gravity cancel inside them near hover), new rates
  d.vx = add2(d.vx, fma2(ua, dvt2, v.dvx));
  d.vy = add2(d.vy, fma2(ub, dvt2, v.dvy));
  d.vz = add2(d.vz, fma2(neg2(uc), dvt2, fma2(0.5f, dvt2, v.dvz)));
  d.wx = fma2(v.Wx, tx, fma2(v.Kx, yz, d.wx));
  d.wy = fma2(v.Wy, ty, fma2(v.Ky, zx, d.wy));
  d.wz = fma2(neg2(v.Wz), tzn, fma2(v.Kz, xy, d.wz));
  d.dx = fma2(u.dt, d.vx, d.dx);
  d.dy = fma2(u.dt, d.vy, d.dy);
  d.dz = fma2(u.dt, d.vz, d.dz);
  // attitude (see above): b = (h + (h^3/3) |w|^2) w
  const V2 wn2 = fma2(d.wx, d.wx, fma2(d.wy, d.wy, mul2(d.wz, d.wz)));
  const V2 sf = fma2(wn2, u.half_dt_cu3, u.half_dt);
  const V2 bx = mul2(sf, d.wx), by = mul2(sf, d.wy), bz = mul2(sf, d.wz);
  const V2 q0 = d.q0, q1 = d.q1, q2 = d.q2, q3 = d.q3;
  V2 n0 = sub2(q0, fma2(q3, bz, fma2(q2, by, mul2(q1, bx))));
  V2 n1 = add2(q1, fma2(neg2(q3), by, fma2(q2, bz, mul2(q0, bx))));
  V2 n2 = add2(q2, fma2(q3, bx, fma2(neg2(q1), bz, mul2(q0, by))));
  V2 n3 = add2(q3, fma2(neg2(q2), bx, fma2(q1, by, mul2(q0, bz))));
  if (!(fmaxf(wn2.x, wn2.y) < u.small_rot_wn2)) {
    if (!(wn2.x < u.small_rot_wn2)) { n0.x = q0.x; n1.x = q1.x; n2.x = q2.x; n3.x = q3.x; quat_step_large(n0.x, n1.x, n2.x, n3.x, d.wx.x, d.wy.x, d.wz.x, wn2.x, u.half_dt); }
    if (!(wn2.y < u.small_rot_wn2)) { n0.y = q0.y; n1.y = q1.y; n2.y = q2.y; n3.y = q3.y; quat_step_large(n0.y, n1.y, n2.y, n3.y, d.wx.y, d.wy.y, d.wz.y, wn2.y, u.half_dt); }
  }
  if constexpr (NORM) {
    const V2 nn = fma2(n0, n0, fma2(n1, n1, fma2(n2, n2, mul2(n3, n3))));
    const V2 rn = fma2(-0.5f, nn, 1.5f);
    d.q0 = mul2(n0, rn); d.q1 = mul2(n1, rn); d.q2 = mul2(n2, rn); d.q3 = mul2(n3, rn);
  } else {
    d.q0 = n0; d.q1 = n1; d.q2 = n2; d.q3 = n3;
  }
}

// The speculative tick (rollout_run_pair): inner_tick_pair<false, LAG> without its two rare paths and without a branch.  It always
// keeps the unclipped mixer outputs and the tan-form quaternion map; a lane where the exact tick would take the rotor-limit path
// (failed sufficient test) or the large-rotation path (|w|^2 >= small_rot_wn2) sets `rare`, and its state is then wrong.
// Where `rare` stays 0 the tick ran exactly the rounded operations of inner_tick_pair<false, LAG>, so the two must change together.
// (A copy rather than a template switch of inner_tick_pair: as a switch, the same operations reach ptxas in another order and the
// speculative kernels compile to different machine code.)
template <bool LAG, class VP> UAVB_DEV void inner_tick_pair_spec(Drone2& d, const VehU<float>& u, const VP& v, unsigned& rare) {
  const V2 yz = mul2(d.wy, d.wz), zx = mul2(d.wz, d.wx), xy = mul2(d.wx, d.wy);
  // mixer butterfly of mix_and_limit_pair, its sufficient test recorded instead of branched on
  const V2 pb = fma2(neg2(v.Jp), d.wx, fma2(v.Gx, yz, d.cp)), qb = fma2(neg2(v.Jq), d.wy, fma2(v.Gy, zx, d.cq));
  const V2 rb = fma2(neg2(v.Jr), d.wz, fma2(v.Gz, xy, d.cr));
  const V2 m1 = add2(pb, qb), m2 = sub2(pb, qb), t1 = add2(d.coll, rb), t2 = sub2(d.coll, rb);
  const V2 need = add2(add2(abs2(pb), abs2(qb)), abs2(rb));
  rare |= (unsigned)(!(need.x <= d.margin.x) | !(need.y <= d.margin.y));
  lag_toward_pair(d, u, sqrt2(add2(t1, m1)), sqrt2(sub2(t2, m2)), sqrt2(sub2(t1, m1)), sqrt2(add2(t2, m2)));
  V2 ha, hb, hc;
  half_axis_pair(d, ha, hb, hc);
  const V2 ua = LAG ? d.zbx : ha, ub = LAG ? d.zby : hb, uc = LAG ? d.zbz : hc;
  d.zbx = ha; d.zby = hb; d.zbz = hc;
  // rotor sums (mujoco_sim.py:235-247): a = s0+s1, c = s0-s1, b = s2+s3, e = s2-s3 with s_i = w_i^2
  const V2 s0 = mul2(d.om0, d.om0), s2 = mul2(d.om2, d.om2);
  const V2 a = fma2(d.om1, d.om1, s0), c = fma2(neg2(d.om1), d.om1, s0);
  const V2 b = fma2(d.om3, d.om3, s2), e = fma2(neg2(d.om3), d.om3, s2);
  const V2 tot = add2(a, b), ty = sub2(a, b), tx = sub2(c, e), tzn = add2(c, e);
  const V2 dvt2 = mul2(neg2(tot), v.kf_dt_over_m2);
  // semi-implicit Euler: velocity increments formed first (thrust and gravity cancel inside them near hover), new rates
  d.vx = add2(d.vx, fma2(ua, dvt2, v.dvx));
  d.vy = add2(d.vy, fma2(ub, dvt2, v.dvy));
  d.vz = add2(d.vz, fma2(neg2(uc), dvt2, fma2(0.5f, dvt2, v.dvz)));
  d.wx = fma2(v.Wx, tx, fma2(v.Kx, yz, d.wx));
  d.wy = fma2(v.Wy, ty, fma2(v.Ky, zx, d.wy));
  d.wz = fma2(neg2(v.Wz), tzn, fma2(v.Kz, xy, d.wz));
  d.dx = fma2(u.dt, d.vx, d.dx);
  d.dy = fma2(u.dt, d.vy, d.dy);
  d.dz = fma2(u.dt, d.vz, d.dz);
  // attitude (see above): b = (h + (h^3/3) |w|^2) w
  const V2 wn2 = fma2(d.wx, d.wx, fma2(d.wy, d.wy, mul2(d.wz, d.wz)));
  const V2 sf = fma2(wn2, u.half_dt_cu3, u.half_dt);
  const V2 bx = mul2(sf, d.wx), by = mul2(sf, d.wy), bz = mul2(sf, d.wz);
  const V2 q0 = d.q0, q1 = d.q1, q2 = d.q2, q3 = d.q3;
  rare |= (unsigned)(!(wn2.x < u.small_rot_wn2) | !(wn2.y < u.small_rot_wn2));
  d.q0 = sub2(q0, fma2(q3, bz, fma2(q2, by, mul2(q1, bx))));
  d.q1 = add2(q1, fma2(neg2(q3), by, fma2(q2, bz, mul2(q0, bx))));
  d.q2 = add2(q2, fma2(q3, bx, fma2(neg2(q1), bz, mul2(q0, by))));
  d.q3 = add2(q3, fma2(neg2(q2), bx, fma2(q1, by, mul2(q0, bz))));
}

// ---------------------------------------------------------------------------------------------
// 100 Hz outer loop of the pair: TrajectoryController._update_outer_loop (main.py:47-61) = altitude (controller.py:26-56),
// lateral (:58-97), roll/pitch (:132-154), yaw (:156-168) on the fresh state, stage by stage as outer_update<float>.

UAVB_DEV V2 rcp2(V2 x) { return make_float2(Math<float>::rcp_fast(x.x), Math<float>::rcp_fast(x.y)); }
UAVB_DEV V2 clamp2(V2 x, float lo, float hi) { return clamp_pair(x, lo, hi); }

// s = limit / |(x, y)| when the norm exceeds the limit, else 1 (multiplying by 1 is exact: the unclamped vector keeps its bits)
UAVB_DEV V2 norm_limit_scale(V2 n2, float limit) {
  const float l2 = __fmul_rn(limit, limit);
  return make_float2(n2.x > l2 ? __fmul_rn(limit, Math<float>::rsqrt(n2.x)) : 1.f, n2.y > l2 ? __fmul_rn(limit, Math<float>::rsqrt(n2.y)) : 1.f);
}

// Math<float>::atan2 for the pair: the polynomial is packed, the reciprocal and the octant / quadrant reflections run per lane.
UAVB_DEV V2 atan2_pair(V2 y, V2 x) {
  const float mx0 = fmaxf(fabsf(x.x), fabsf(y.x)), mn0 = fminf(fabsf(x.x), fabsf(y.x));
  const float mx1 = fmaxf(fabsf(x.y), fabsf(y.y)), mn1 = fminf(fabsf(x.y), fabsf(y.y));
  const V2 a = make_float2(mx0 > 0.f ? __fmul_rn(mn0, Math<float>::rcp_fast(mx0)) : 0.f, mx1 > 0.f ? __fmul_rn(mn1, Math<float>::rcp_fast(mx1)) : 0.f);
  const V2 t = mul2(a, a);
  V2 p = fma2(-0.0040545563519447094f, t, 0.02186292376737154f);
  p = fma2(p, t, -0.055912287992173626f);
  p = fma2(p, t, 0.09642195584271772f);
  p = fma2(p, t, -0.13908629508211973f);
  p = fma2(p, t, 0.19946565845760894f);
  p = fma2(p, t, -0.33329860832632324f);
  p = fma2(p, t, 0.9999993356075512f);
  const V2 r = mul2(a, p);
  float r0 = r.x, r1 = r.y;
  r0 = (fabsf(y.x) > fabsf(x.x)) ? __fadd_rn(1.57079632679489662f, -r0) : r0;
  r1 = (fabsf(y.y) > fabsf(x.y)) ? __fadd_rn(1.57079632679489662f, -r1) : r1;
  r0 = (x.x < 0.f) ? __fadd_rn(3.14159265358979324f, -r0) : r0;
  r1 = (x.y < 0.f) ? __fadd_rn(3.14159265358979324f, -r1) : r1;
  return make_float2(copysignf(r0, y.x), copysignf(r1, y.y));
}

// Per-rollout constants of the outer loop for the pair (gains and mass).
struct VehO2 {
  V2 mass, kp_xy, kd_xy, kp_z, kd_z, ki_z, kp_roll, kp_pitch, kp_yaw, Jp, Jq, Jr;
};
UAVB_DEV void zip_veho(VehO2& o, const VehP<float>& a, const VehP<float>& b) {
  o.mass = make_float2(a.mass, b.mass); o.kp_xy = make_float2(a.kp_xy, b.kp_xy); o.kd_xy = make_float2(a.kd_xy, b.kd_xy);
  o.kp_z = make_float2(a.kp_z, b.kp_z); o.kd_z = make_float2(a.kd_z, b.kd_z); o.ki_z = make_float2(a.ki_z, b.ki_z);
  o.kp_roll = make_float2(a.kp_roll, b.kp_roll); o.kp_pitch = make_float2(a.kp_pitch, b.kp_pitch); o.kp_yaw = make_float2(a.kp_yaw, b.kp_yaw);
  o.Jp = make_float2(a.Jp, b.Jp); o.Jq = make_float2(a.Jq, b.Jq); o.Jr = make_float2(a.Jr, b.Jr);
}

// Set-point of the pair: fields are V2 (per-lane missions) or float (shared mission: one row for both lanes).
template <class T> struct Target2 {
  T vx, vy, vz, ax, ay, az, yc, ys;
};

// (ex, ey, ez) = set-point - position, formed in fp64 per lane by the caller and rounded once.
template <class T> UAVB_DEV void outer_update_pair(Drone2& d, const VehU<float>& u, const VehO2& v, const Target2<T>& t, V2 ex, V2 ey, V2 ez) {
  const V2 q0 = d.q0, q1 = d.q1, q2 = d.q2, q3 = d.q3;
  // products of R(q) (quad.py:153, unit quaternion): h_ij = R_ij / 2 off the diagonal, d_ii = (1 - R_ii) / 2
  const V2 q11 = mul2(q1, q1), q22 = mul2(q2, q2), q33 = mul2(q3, q3);
  const V2 R00 = fma2(-2.f, add2(q22, q33), 1.f), R11 = fma2(-2.f, add2(q11, q33), 1.f), R22 = fma2(-2.f, add2(q11, q22), 1.f);
  const V2 q12 = mul2(q1, q2), q13 = mul2(q1, q3), q23 = mul2(q2, q3);
  const V2 R01 = mul2(2.f, fma2(neg2(q0), q3, q12)), R10 = mul2(2.f, fma2(q0, q3, q12));
  const V2 R02 = mul2(2.f, fma2(q0, q2, q13)), R12 = mul2(2.f, fma2(neg2(q0), q1, q23));
  const V2 sa = mul2(2.f, fma2(q0, q1, q23));                          // R21 = sin(phi) cos(theta)
  const V2 inv_R22 = rcp2(R22);
  // altitude (controller.py:26-56)
  const V2 climb = clamp2(as2(t.vz), -u.max_ascent, u.max_descent);
  const V2 ezd = sub2(climb, d.vz);
  const V2 integ = clamp2(fma2(ez, u.dt_outer, make_float2(d.integral[0], d.integral[1])), -u.integral_limit, u.integral_limit);
  d.integral[0] = integ.x; d.integral[1] = integ.y;
  V2 acc_z = fma2(v.kp_z, ez, fma2(v.ki_z, integ, fma2(v.kd_z, ezd, sub2(as2(t.az), u.g))));
  acc_z = mul2(acc_z, inv_R22);
  const V2 c = clamp2(mul2(neg2(v.mass), acc_z), u.fmin4, u.fmax4);
  d.thrust_cmd[0] = c.x; d.thrust_cmd[1] = c.y;
  d.coll = mul2(u.quarter_inv_kf, c);                                // c is already inside [4 fmin, 4 fmax] (quad.py:107,113)
  d.margin = make_float2(limit_margin(d.coll.x, u.w2min, u.w2max), limit_margin(d.coll.y, u.w2min, u.w2max));
  // lateral (controller.py:58-97)
  V2 vxd = as2(t.vx), vyd = as2(t.vy);
  const V2 sv = norm_limit_scale(fma2(vxd, vxd, mul2(vyd, vyd)), u.max_speed_xy);
  vxd = mul2(vxd, sv); vyd = mul2(vyd, sv);
  V2 ax = fma2(v.kp_xy, ex, fma2(v.kd_xy, sub2(vxd, d.vx), t.ax));
  V2 ay = fma2(v.kp_xy, ey, fma2(v.kd_xy, sub2(vyd, d.vy), t.ay));
  const V2 sacc = norm_limit_scale(fma2(ax, ax, mul2(ay, ay)), u.max_acc_xy);
  ax = mul2(ax, sacc); ay = mul2(ay, sacc);
  const V2 inv_accz = mul2(neg2(v.mass), rcp2(c));                    // 1 / (-c/m)
  const V2 bx = clamp2(mul2(ax, inv_accz), -u.max_tilt, u.max_tilt), by = clamp2(mul2(ay, inv_accz), -u.max_tilt, u.max_tilt);
  // roll / pitch (controller.py:132-154)
  const V2 bdx = mul2(v.kp_roll, sub2(bx, R02)), bdy = mul2(v.kp_pitch, sub2(by, R12));
  const V2 p_c = mul2(fma2(R10, bdx, neg2(mul2(R00, bdy))), inv_R22);
  const V2 q_c = mul2(fma2(R11, bdx, neg2(mul2(R01, bdy))), inv_R22);
  // yaw (controller.py:156-168), unit-quaternion form of yaw_rate_cmd_unit: sp = R10, cp = R00
  const V2 e_yaw = atan2_pair(fma2(t.ys, R00, neg2(mul2(t.yc, R10))), fma2(t.yc, R00, mul2(t.ys, R10)));
  const V2 ct2 = fma2(sa, sa, mul2(R22, R22));                       // cos(theta)^2
  const V2 r_c = mul2(fma2(mul2(v.kp_yaw, e_yaw), ct2, neg2(mul2(q_c, sa))), inv_R22);
  d.cp = mul2(v.Jp, p_c); d.cq = mul2(v.Jq, q_c); d.cr = mul2(v.Jr, r_c);
}

}  // namespace uavb
