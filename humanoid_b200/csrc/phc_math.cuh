// Device-side quaternion / frame-blend arithmetic of the PHC step path (sm_100a).
//
// Every function reproduces the fp32 operation ORDER of the reference primitive it cites
// (paths relative to packages/puffer-phc/puffer_phc/), because two places on the path are
// rounding-sensitive: the frame index is a truncation of a value that lands on integers
// (motion_lib.py:661), and slerp's sqrt(1 - c*c) cancels catastrophically for consecutive
// mocap frames (torch_utils.py:121).  This translation unit is compiled with -fmad=false so
// a*b+c is two roundings, as in ATen's one-kernel-per-op evaluation; the two places where
// ATen's CPU kernels do fuse (cross product, 3-vector norm) use __fmaf_rn explicitly.
// The integer path (calc_frame_blend) and everything a termination flag depends on use IEEE
// division / square root (-prec-div/-prec-sqrt default, no fast-math).  The float-only outputs
// use branch-free "faithful" (<= 1-2 ulp) replacements where the reference's value is itself a
// rounded transcendental: see sin_q1 / sqrt_faithful / div_faithful / wrap_angle below and
// DESIGN.md "arithmetic" for the measured effect (1e-7 relative, against the 1e-5 tolerance).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace phc {

struct Vec3 {
  float x, y, z;
};
struct Quat {
  float x, y, z, w;
};

__device__ __forceinline__ Vec3 operator-(Vec3 a, Vec3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ Vec3 operator+(Vec3 a, Vec3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }

// torch.clip(x, 0, 1) on finite input; NaN maps to 0 (the reference would index out of range)
__device__ __forceinline__ float clip01(float x) { return fminf(fmaxf(x, 0.0f), 1.0f); }

// ---- branch-free faithful primitives (float outputs only) -----------------------------------
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// a / b given r ~ 1/b: one Newton correction of the quotient, <= 1 ulp, no special-case path
__device__ __forceinline__ float div_faithful(float a, float b, float r) {
  const float q = a * r;
  return __fmaf_rn(__fmaf_rn(-b, q, a), r, q);
}
// sqrt(x) for normal x > 0 (NaN for x <= 0, which every caller masks afterwards)
__device__ __forceinline__ float sqrt_faithful(float x) {
  const float r = rsqrt_approx(x);
  const float s = x * r;
  return __fmaf_rn(__fmaf_rn(-s, s, x), 0.5f * r, s);
}
// sin(x) on [0, pi/2] (slerp's arguments are t*theta with theta = acos(|c|) <= pi/2): odd minimax
// polynomial x + x^3 q(x^2), <= 1.7 ulp, 87 % correctly rounded (profiles/sin_poly_fit.py); no range
// reduction and no Payne-Hanek slow path, unlike sinf.
__device__ __forceinline__ float sin_q1(float x) {
  const float u = x * x;
  float q = 2.6018724383902736e-06f;
  q = __fmaf_rn(q, u, -0.00019807404896710068f);
  q = __fmaf_rn(q, u, 0.008333024568855762f);
  q = __fmaf_rn(q, u, -0.16666656732559204f);
  return __fmaf_rn(x * u, q, x);
}
// normalize_angle(a) = atan2(sin a, cos a) (torch_utils.py:50-51) for a in [0, 2 pi]: the wrap to
// (-pi, pi] it computes, without the three transcendentals.  ATen's own evaluation is within
// 2.4e-7 absolute of this (measured over 6M angles), i.e. at the level of its rounding noise.
__device__ __forceinline__ float wrap_angle_0_2pi(float a) {
  return a > 3.14159274101257324f ? a - 6.28318548202514648f : a;
}

// MotionLibBase._calc_frame_blend, motion_lib.py:655-665.
//   phase = clip(t / len, 0, 1)   (from the un-clamped time)
//   t[t < 0] = 0
//   idx0 = trunc(phase * f32(nf - 1)); idx1 = min(idx0 + 1, nf - 1)
//   blend = clip((t - f32(idx0) * dt) / dt, 0, 1)
__device__ __forceinline__ void calc_frame_blend(float t, float len, int64_t nf, float dt, int64_t& idx0,
                                                 int64_t& idx1, float& blend) {
  float phase = clip01(t / len);
  if (t < 0.0f) t = 0.0f;
  idx0 = (int64_t)(phase * (float)(nf - 1));
  idx1 = idx0 + 1 < nf - 1 ? idx0 + 1 : nf - 1;
  blend = clip01((t - (float)idx0 * dt) / dt);
}

// The same with 32-bit frame counts (any clip below 2^31 frames): identical results — int32 and
// int64 convert to the same float, and the truncation is of a value in [0, nf-1].
__device__ __forceinline__ void calc_frame_blend32(float t, float len, int nf, float dt, int& idx0, int& idx1,
                                                   float& blend) {
  float phase = clip01(t / len);
  if (t < 0.0f) t = 0.0f;
  idx0 = (int)(phase * (float)(nf - 1));
  idx1 = idx0 + 1 < nf - 1 ? idx0 + 1 : nf - 1;
  blend = clip01((t - (float)idx0 * dt) / dt);
}

// quat_mul, torch_utils.py:55-75.  The reference uses an 8-multiply form whose absolute error is
// ~1e-7 for unit quaternions; the Hamilton product accumulated with FMAs has the same error level
// in 16 instructions instead of 26, so it is used for every product on the path (the operands are
// slerp outputs that already differ from the reference's by their sin/acos rounding).
__device__ __forceinline__ Quat quat_mul(Quat a, Quat b) {
  Quat r;
  r.x = __fmaf_rn(a.w, b.x, __fmaf_rn(a.x, b.w, __fmaf_rn(a.y, b.z, -(a.z * b.y))));
  r.y = __fmaf_rn(a.w, b.y, __fmaf_rn(a.y, b.w, __fmaf_rn(a.z, b.x, -(a.x * b.z))));
  r.z = __fmaf_rn(a.w, b.z, __fmaf_rn(a.z, b.w, __fmaf_rn(a.x, b.y, -(a.y * b.x))));
  r.w = __fmaf_rn(a.w, b.w, -__fmaf_rn(a.x, b.x, __fmaf_rn(a.y, b.y, a.z * b.z)));
  return r;
}

__device__ __forceinline__ Quat quat_conj(Quat q) { return {-q.x, -q.y, -q.z, q.w}; }

// w of quat_mul(a, conj(b)) — all the reward needs of the rotation difference (common.py:304-306)
__device__ __forceinline__ float quat_mul_conj_w(Quat a, Quat b) {
  return __fmaf_rn(a.w, b.w, __fmaf_rn(a.x, b.x, __fmaf_rn(a.y, b.y, a.z * b.z)));
}

// A heading quaternion (0, 0, z, w): rotation about the up axis.  The x, y components of
// calc_heading_quat(_inv) are exactly +-0 (torch_utils.py:354-358 with axis (0,0,1)), so the
// products below only keep the terms that survive.
struct Heading {
  float z, w;
};

// quat_mul(h, q) with h = (0,0,z,w)
__device__ __forceinline__ Quat heading_mul_left(Heading h, Quat b) {
  Quat r;
  r.x = __fmaf_rn(h.w, b.x, -(h.z * b.y));
  r.y = __fmaf_rn(h.w, b.y, h.z * b.x);
  r.z = __fmaf_rn(h.w, b.z, h.z * b.w);
  r.w = __fmaf_rn(h.w, b.w, -(h.z * b.z));
  return r;
}

// quat_mul(q, h) with h = (0,0,z,w)
__device__ __forceinline__ Quat heading_mul_right(Quat a, Heading h) {
  Quat r;
  r.x = __fmaf_rn(a.x, h.w, a.y * h.z);
  r.y = __fmaf_rn(a.y, h.w, -(a.x * h.z));
  r.z = __fmaf_rn(a.z, h.w, a.w * h.z);
  r.w = __fmaf_rn(a.w, h.w, -(a.z * h.z));
  return r;
}

// my_quat_rotate, torch_utils.py:274-281, with q = (0,0,z,w):
//   x' = x(2w^2-1) - 2zw y,   y' = y(2w^2-1) + 2zw x,   z' = z((2w^2-1) + 2z^2)
// The three coefficients are formed once per thread.
struct HeadingRot {
  float a, b, d;
};
__device__ __forceinline__ HeadingRot heading_rot(Heading h) {
  HeadingRot c;
  c.a = __fmaf_rn(2.0f * h.w, h.w, -1.0f);
  c.b = 2.0f * h.z * h.w;
  c.d = __fmaf_rn(2.0f * h.z, h.z, c.a);
  return c;
}
__device__ __forceinline__ Vec3 heading_rotate(const HeadingRot& c, Vec3 v) {
  return {__fmaf_rn(v.x, c.a, -(v.y * c.b)), __fmaf_rn(v.y, c.a, v.x * c.b), v.z * c.d};
}

// quat_to_tan_norm, torch_utils.py:285-297: my_quat_rotate of (1,0,0) and of (0,0,1):
//   tan  = (2w^2-1 + 2x^2,  2zw + 2xy,  -2yw + 2xz),   norm = (2yw + 2xz,  -2xw + 2yz,  2w^2-1 + 2z^2)
__device__ __forceinline__ void quat_tan_norm(Quat q, float* out6) {
  const float x2 = q.x + q.x, y2 = q.y + q.y, z2 = q.z + q.z;
  const float s = __fmaf_rn(q.w + q.w, q.w, -1.0f);
  out6[0] = __fmaf_rn(x2, q.x, s);
  out6[1] = __fmaf_rn(z2, q.w, y2 * q.x);
  out6[2] = __fmaf_rn(z2, q.x, -(y2 * q.w));
  out6[3] = __fmaf_rn(y2, q.w, x2 * q.z);
  out6[4] = __fmaf_rn(y2, q.z, -(x2 * q.w));
  out6[5] = __fmaf_rn(z2, q.z, s);
}

// remove_base_rot, envs/common.py:15-19: q (x) conj(0.5,0.5,0.5,0.5)
__device__ __forceinline__ Quat remove_base_rot(Quat q) { return quat_mul(q, Quat{-0.5f, -0.5f, -0.5f, 0.5f}); }

// calc_heading_quat_inv / calc_heading_quat, torch_utils.py:369-408.
//   heading = atan2(rot.y, rot.x), rot = my_quat_rotate(q,(1,0,0))
//   q_h = quat_unit((0,0,sin(+-heading/2), cos(heading/2)))   (norm: sequential, no FMA)
// heading_quat == conj(heading_quat_inv) exactly, so one evaluation serves both.
__device__ __forceinline__ Heading heading_quat_inv(Quat q) {
  float s = 2.0f * (q.w * q.w) - 1.0f;
  float rx = s + q.x * q.x * 2.0f;
  float ry = q.z * q.w * 2.0f + q.y * q.x * 2.0f;
  float half = (-atan2f(ry, rx)) / 2.0f;
  float sn = sinf(half), cs = cosf(half);
  float nrm = fmaxf(sqrtf(sn * sn + cs * cs), 1e-9f);
  return {sn / nrm, cs / nrm};
}
__device__ __forceinline__ Heading heading_conj(Heading h) { return {-h.z, h.w}; }

// angle of quat_to_angle_axis, torch_utils.py:86-106:
//   sin_theta = sqrt(1 - w*w); angle = normalize_angle(2*acos(w)); 0 unless |sin_theta| > 1e-5.
// The mask is evaluated on 1 - w*w directly (sqrt is monotonic; |w| > 1 gives a negative or NaN
// argument and the comparison is false, as abs(NaN) > 1e-5 is in the reference).
__device__ __forceinline__ float quat_angle(float w) {
  const float x = 1.0f - w * w;
  const float a = wrap_angle_0_2pi(2.0f * acosf(w));
  return (x > 1.0000000e-10f) ? a : 0.0f;
}

// quat_to_exp_map, torch_utils.py:135-150 (only get_motion_state's dof_pos needs the axis)
__device__ __forceinline__ Vec3 quat_exp_map(Quat q) {
  const float st = sqrtf(1.0f - q.w * q.w);
  const float a = wrap_angle_0_2pi(2.0f * acosf(q.w));
  if (fabsf(st) > 1e-5f) return {a * (q.x / st), a * (q.y / st), a * (q.z / st)};
  return {0.0f, 0.0f, 0.0f};
}

// torch.norm(v, dim=-1) over 3 on ATen CPU: sqrt(fma(z,z,fma(y,y,x*x)))
__device__ __forceinline__ float norm3(Vec3 v) { return sqrtf(__fmaf_rn(v.z, v.z, __fmaf_rn(v.y, v.y, v.x * v.x))); }

// exp_map_to_quat, torch_utils.py:334-366: angle = |e| wrapped to (-pi, pi] by atan2(sin, cos), axis
// e/|e| (z axis when |angle| <= 1e-5), then quat_from_angle_axis incl. its two normalisations
__device__ __forceinline__ Quat exp_map_to_quat(Vec3 e) {
  float ang = norm3(e);
  Vec3 ax = {e.x / ang, e.y / ang, e.z / ang};
  ang = atan2f(sinf(ang), cosf(ang));
  if (!(fabsf(ang) > 1e-5f)) {
    ang = 0.0f;
    ax = {0.0f, 0.0f, 1.0f};
  }
  const float an = fmaxf(norm3(ax), 1e-9f);
  const float half = ang / 2.0f;
  const float sn = sinf(half), cs = cosf(half);
  Quat q = {ax.x / an * sn, ax.y / an * sn, ax.z / an * sn, cs};
  const float qn = fmaxf(sqrtf(((q.x * q.x + q.y * q.y) + q.z * q.z) + q.w * q.w), 1e-9f);
  return {q.x / qn, q.y / qn, q.z / qn, q.w / qn};
}

// slerp, torch_utils.py:110-131.  c = ((x0x1 + y0y1) + z0z1) + w0w1 (ATen sum order);
// q1 flipped when c < 0; result not renormalised; the |sin| < 1e-3 average is applied
// first and the |cos| >= 1 -> q0 select last (it wins, and masks acos' NaN for c > 1).
__device__ __forceinline__ Quat quat_slerp(Quat q0, Quat q1, float t) {
  float c = ((q0.x * q1.x + q0.y * q1.y) + q0.z * q1.z) + q0.w * q1.w;
  const float sg = c < 0.0f ? -1.0f : 1.0f;  // q1[neg] = -q1[neg]: folded into q1's coefficient
  c = fabsf(c);
  const float th = acosf(c);
  const float s = sqrt_faithful(1.0f - c * c);  // 1 - c*c: two roundings, never an FMA
  const float rs = rcp_approx(s);
  float ra = div_faithful(sin_q1((1.0f - t) * th), s, rs);
  float rb = div_faithful(sin_q1(t * th), s, rs);
  const bool avg = fabsf(s) < 0.001f;  // false for NaN, as in the reference
  ra = avg ? 0.5f : ra;                // 0.5 q0 + 0.5 q1
  rb = avg ? 0.5f : rb;
  const bool same = c >= 1.0f;         // -> q0; applied last, masks the NaNs of acos(c > 1)
  ra = same ? 1.0f : ra;
  rb = (same ? 0.0f : rb) * sg;
  return {__fmaf_rn(rb, q1.x, ra * q0.x), __fmaf_rn(rb, q1.y, ra * q0.y), __fmaf_rn(rb, q1.z, ra * q0.z),
          __fmaf_rn(rb, q1.w, ra * q0.w)};
}

// lerp of get_motion_state, motion_lib.py:597-603: (1 - b)*x0 + b*x1
__device__ __forceinline__ Vec3 lerp3(float om, float b, Vec3 x0, Vec3 x1) {
  return {om * x0.x + b * x1.x, om * x0.y + b * x1.y, om * x0.z + b * x1.z};
}

// (d**2).mean(dim=-1) over 3: ((x^2 + y^2) + z^2) / 3, the division as a multiply by fl(1/3)
// (<= 1 ulp from the quotient; feeds only the reward's exponent)
__device__ __forceinline__ float mean_sq3(Vec3 d) {
  return __fmaf_rn(d.z, d.z, __fmaf_rn(d.y, d.y, d.x * d.x)) * 0.333333343267440796f;
}

// ---- packed fp32x2 (sm_100: FFMA2 / FMUL2) -----------------------------------------------------------------------
// Two independent evaluations of the same operation sequence in one instruction; each lane is rounded exactly as the
// scalar instruction is, so lane k of every *x2 helper below equals the scalar helper it names, bit for bit.
// ptxas fuses a packed multiply followed by a packed add into one FFMA2 even under -fmad=false (CUDA 12.9), which would
// round a lerp once less than the reference.  So the packed add is an FMA by `one`, a 1.0f the compiler cannot see
// (a kernel parameter): p * 1 is exact, so each lane is rn(p + q) for every input, ±0, subnormals, inf and NaN included,
// and ptxas leaves the multiply that produced p alone.  Check new uses in SASS (profiles/sass_mix.py).
struct Vec3x2 {
  float2 x, y, z;
};
struct Quatx2 {
  float2 x, y, z, w;
};
__device__ __forceinline__ float2 bc2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 add2(float2 a, float2 b, float one) { return __ffma2_rn(a, bc2(one), b); }
// a - b as rn(b * -1 + a)
__device__ __forceinline__ float2 sub2(float2 a, float2 b, float one) { return __ffma2_rn(b, bc2(-one), a); }

__device__ __forceinline__ Vec3x2 pack3(Vec3 a, Vec3 b) { return {{a.x, b.x}, {a.y, b.y}, {a.z, b.z}}; }
__device__ __forceinline__ Quatx2 pack4(Quat a, Quat b) { return {{a.x, b.x}, {a.y, b.y}, {a.z, b.z}, {a.w, b.w}}; }
__device__ __forceinline__ Vec3 lane0(Vec3x2 v) { return {v.x.x, v.y.x, v.z.x}; }
__device__ __forceinline__ Vec3 lane1(Vec3x2 v) { return {v.x.y, v.y.y, v.z.y}; }

// lane k equals a - b (Vec3 operator-) bit for bit
__device__ __forceinline__ Vec3x2 sub3x2(Vec3x2 a, Vec3x2 b, float one) {
  return {sub2(a.x, b.x, one), sub2(a.y, b.y, one), sub2(a.z, b.z, one)};
}
// lane k equals lerp3 bit for bit
__device__ __forceinline__ Vec3x2 lerp3x2(float2 om, float2 b, Vec3x2 x0, Vec3x2 x1, float one) {
  return {add2(mul2(om, x0.x), mul2(b, x1.x), one), add2(mul2(om, x0.y), mul2(b, x1.y), one),
          add2(mul2(om, x0.z), mul2(b, x1.z), one)};
}
// lane k equals sin_q1 bit for bit
__device__ __forceinline__ float2 sin_q1x2(float2 x) {
  const float2 u = mul2(x, x);
  float2 q = fma2(u, bc2(2.6018724383902736e-06f), bc2(-0.00019807404896710068f));
  q = fma2(q, u, bc2(0.008333024568855762f));
  q = fma2(q, u, bc2(-0.16666656732559204f));
  return fma2(mul2(x, u), q, x);
}
// lane k equals div_faithful bit for bit
__device__ __forceinline__ float2 div_faithful2(float2 a, float2 b, float2 r) {
  const float2 q = mul2(a, r);
  return fma2(fma2(neg2(b), q, a), r, q);
}
// the per-lane part of quat_slerp: the sign fold, acos, the MUFU approximations and the select chain's inputs
__device__ __forceinline__ void slerp_lane(float c, float& sg, float& ca, float& th, float& s, float& rs) {
  sg = c < 0.0f ? -1.0f : 1.0f;
  ca = fabsf(c);
  th = acosf(ca);
  s = sqrt_faithful(1.0f - ca * ca);
  rs = rcp_approx(s);
}
__device__ __forceinline__ void slerp_select(float ca, float s, float sg, float& ra, float& rb) {
  const bool avg = fabsf(s) < 0.001f;
  ra = avg ? 0.5f : ra;
  rb = avg ? 0.5f : rb;
  const bool same = ca >= 1.0f;
  ra = same ? 1.0f : ra;
  rb = (same ? 0.0f : rb) * sg;
}
// (x, y) and (z, w) of a quaternion as they arrive from one 16-byte load: already register pairs
__device__ __forceinline__ float2 qxy(Quat q) { return make_float2(q.x, q.y); }
__device__ __forceinline__ float2 qzw(Quat q) { return make_float2(q.z, q.w); }
// quat_slerp's c, ((x0x1 + y0y1) + z0z1) + w0w1, with the four products as two packed multiplies
__device__ __forceinline__ float slerp_dot(Quat q0, Quat q1) {
  const float2 xy = mul2(qxy(q0), qxy(q1)), zw = mul2(qzw(q0), qzw(q1));
  return ((xy.x + xy.y) + zw.x) + zw.y;
}
// ra * q0 + rb * q1 componentwise, as quat_slerp's last line: __fmaf_rn(rb, q1.c, ra * q0.c)
__device__ __forceinline__ Quat slerp_mix(Quat q0, Quat q1, float ra, float rb) {
  const float2 xy = fma2(qxy(q1), bc2(rb), mul2(qxy(q0), bc2(ra)));
  const float2 zw = fma2(qzw(q1), bc2(rb), mul2(qzw(q0), bc2(ra)));
  return {xy.x, xy.y, zw.x, zw.y};
}
// Two slerps at once: out0 equals quat_slerp(a0, a1, t.x) and out1 quat_slerp(b0, b1, t.y), bit for bit.  The dot
// products and the final mix pair the components of one quaternion; sin and the quotient pair the two slerps.
__device__ __forceinline__ void quat_slerp_pair(Quat a0, Quat a1, Quat b0, Quat b1, float2 t, Quat& out0, Quat& out1) {
  float2 sg, ca, th, s, rs;
  slerp_lane(slerp_dot(a0, a1), sg.x, ca.x, th.x, s.x, rs.x);
  slerp_lane(slerp_dot(b0, b1), sg.y, ca.y, th.y, s.y, rs.y);
  const float2 om = {1.0f - t.x, 1.0f - t.y};
  float2 ra = div_faithful2(sin_q1x2(mul2(om, th)), s, rs);
  float2 rb = div_faithful2(sin_q1x2(mul2(t, th)), s, rs);
  slerp_select(ca.x, s.x, sg.x, ra.x, rb.x);
  slerp_select(ca.y, s.y, sg.y, ra.y, rb.y);
  out0 = slerp_mix(a0, a1, ra.x, rb.x);
  out1 = slerp_mix(b0, b1, ra.y, rb.y);
}
// lane k equals heading_mul_left(h, lane k of b) bit for bit (-(h.z * y) = (-h.z) * y exactly)
__device__ __forceinline__ Quatx2 heading_mul_left2(Heading h, Quatx2 b) {
  const float2 w = bc2(h.w), z = bc2(h.z), nz = bc2(-h.z);
  return {fma2(b.x, w, mul2(b.y, nz)), fma2(b.y, w, mul2(b.x, z)), fma2(b.z, w, mul2(b.w, z)), fma2(b.w, w, mul2(b.z, nz))};
}
// lane k equals heading_rotate(c, lane k of v) bit for bit
__device__ __forceinline__ Vec3x2 heading_rotate2(const HeadingRot& c, Vec3x2 v) {
  return {fma2(v.x, bc2(c.a), mul2(v.y, bc2(-c.b))), fma2(v.y, bc2(c.a), mul2(v.x, bc2(c.b))), mul2(v.z, bc2(c.d))};
}
// lane k of out6[i] equals quat_tan_norm(lane k of q)[i] bit for bit
__device__ __forceinline__ void quat_tan_norm2(Quatx2 q, float one, float2* out6) {
  const float2 x2 = add2(q.x, q.x, one), y2 = add2(q.y, q.y, one), z2 = add2(q.z, q.z, one);
  const float2 s = fma2(add2(q.w, q.w, one), q.w, bc2(-1.0f));
  const float2 nw = neg2(q.w);
  out6[0] = fma2(x2, q.x, s);
  out6[1] = fma2(z2, q.w, mul2(y2, q.x));
  out6[2] = fma2(z2, q.x, mul2(y2, nw));
  out6[3] = fma2(y2, q.w, mul2(x2, q.z));
  out6[4] = fma2(y2, q.z, mul2(x2, nw));
  out6[5] = fma2(z2, q.z, s);
}

// ATen CPU sum over a contiguous row of n floats (aten/src/ATen/native/cpu/SumKernel.cpp, the AVX2 build that torch
// dispatches to on AVX2 and AVX-512 hosts alike; checked against torch 2.11 for every n in 1..48, tests/test_oracle_c.py):
//   n >= 8  vectorized_inner_sum: the n / 8 full vectors are added lane-wise in order (lane l = v[l] + v[l+8] + ..),
//           then the scalar accumulator takes the n % 8 tail elements FIRST, in order, and the 8 lanes after them;
//   n <  8  scalar_inner_sum -> row_sum with four partials: p[k] = v[k] (k < 4), the elements from 4 on go to p[0],
//           then ((p0 + p1) + p2) + p3.
// Valid for n <= 39 (from 5 vectors on ATen's four-way unrolling reorders the lane sums).
__device__ __forceinline__ float aten_row_sum(const float* v, int n) {
  if (n < 8) {
    float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;  // 0 + x is exact
    if (n >= 4) {
      p0 = v[0], p1 = v[1], p2 = v[2], p3 = v[3];
      for (int i = 4; i < n; ++i) p0 += v[i];
    } else {
      for (int i = 0; i < n; ++i) p0 += v[i];
    }
    return ((p0 + p1) + p2) + p3;
  }
  const int nv = n >> 3;
  float acc[8];
#pragma unroll
  for (int l = 0; l < 8; ++l) acc[l] = v[l];
  for (int i = 1; i < nv; ++i) {
#pragma unroll
    for (int l = 0; l < 8; ++l) acc[l] += v[i * 8 + l];
  }
  float s = 0.0f;
  for (int k = nv * 8; k < n; ++k) s += v[k];
#pragma unroll
  for (int l = 0; l < 8; ++l) s = s + acc[l];
  return s;
}

__device__ __forceinline__ float row_sum24(const float* v) {
  float acc[8];
#pragma unroll
  for (int l = 0; l < 8; ++l) acc[l] = (v[l] + v[l + 8]) + v[l + 16];
  float s = acc[0];
#pragma unroll
  for (int l = 1; l < 8; ++l) s = s + acc[l];
  return s;
}

}  // namespace phc
