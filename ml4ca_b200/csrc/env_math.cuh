// env_math.cuh -- per-environment device arithmetic of the ReVolt gym wrapper and the stand-in hull.
//
// Everything here is a __device__ __forceinline__ function on scalars so that the stand-alone env-step kernel
// (env_step.cu) and the fused policy+env rollout kernel (rollout.cu) share one implementation.
// Reference: /root/reference/src/rl/windows_workspace/specific/customEnv.py (cited per function).
//
// Floating point contract (tests/test_env_parity.py):
//  * integer / compare logic -- clip saturation decisions, termination flags, episode counters, the
//    action -> thruster index map -- is bit-exact;
//  * products/quotients that the reference evaluates with one operation (a*bound, prev_thrust/100) use the
//    _rn intrinsics so that no FMA contraction changes the rounding: they equal the float32 oracle bit for bit;
//  * transcendental pieces (atan2f, sincosf, expf, sqrtf chains) carry a stated tolerance against float64.
#pragma once
#include <stdint.h>

#include "ml4ca_constants.h"
#include "philox.cuh"

namespace ml4ca {

constexpr float kPi = (float)ML4CA_PI;

// ---- static description of the four reference env classes ---------------------------------------------------
// ACT  : network action dim           NCMD : real commands after the angle transform (customEnv.py:47-53)
// NANG : azimuths that are per-env state (the others are constants of the class)
template <int KIND, bool CONT>
struct EnvTraits;
template <bool CONT>
struct EnvTraits<ML4CA_ENV_FULL, CONT> {  // customEnv.py:58-65
  static constexpr int ACT = 6, NCMD = 6, NANG = 3;
  static constexpr float ANG_BOUND = kPi;
  static constexpr float DEF_BOW = 0.f, DEF_PORT = 0.f, DEF_STAR = 0.f;
};
template <bool CONT>
struct EnvTraits<ML4CA_ENV_SIMPLE, CONT> {  // customEnv.py:331-349
  static constexpr int ACT = 3, NCMD = 3, NANG = 0;
  static constexpr float ANG_BOUND = kPi;  // unused
  static constexpr float DEF_BOW = (float)(ML4CA_PI / 2), DEF_PORT = (float)(-3 * ML4CA_PI / 4),
                         DEF_STAR = (float)(3 * ML4CA_PI / 4);
};
template <bool CONT>
struct EnvTraits<ML4CA_ENV_LIMITED, CONT> {  // customEnv.py:355-371
  static constexpr int ACT = 5, NCMD = 5, NANG = 2;
  static constexpr float ANG_BOUND = (float)(ML4CA_PI / 2);
  static constexpr float DEF_BOW = (float)(ML4CA_PI / 2), DEF_PORT = 0.f, DEF_STAR = 0.f;
};
template <bool CONT>
struct EnvTraits<ML4CA_ENV_FINAL, CONT> {  // customEnv.py:377-399
  static constexpr int ACT = CONT ? 7 : 5, NCMD = 5, NANG = 2;
  static constexpr float ANG_BOUND = kPi;
  static constexpr float DEF_BOW = (float)(ML4CA_PI / 2), DEF_PORT = 0.f, DEF_STAR = 0.f;
};

// ---- mathematics.py:14-17 ------------------------------------------------------------------------------------
// wrap_angle(a, deg=False): mod(a + pi, 2 pi) - pi with Python's sign-of-divisor modulo.
__device__ __forceinline__ float wrap_rad(float a) {
  const float two_pi = __fmul_rn(2.0f, kPi);
  const float x = __fadd_rn(a, kPi);
  float m = fmodf(x, two_pi);
  if (m < 0.f) m = __fadd_rn(m, two_pi);
  return __fsub_rn(m, kPi);
}
// wrap_angle(a) with its default deg=True applied to RADIAN inputs (errorFrame.py:29,31): the identity for
// -180 <= a < 180, where evaluating (a + 180) mod 360 - 180 literally in fp32 would only inject ~1e-5 noise.
__device__ __forceinline__ float wrap_deg_quirk(float a) {
  if (a >= -180.f && a < 180.f) return a;
  const float x = __fadd_rn(a, 180.f);
  float m = fmodf(x, 360.f);
  if (m < 0.f) m = __fadd_rn(m, 360.f);
  return __fsub_rn(m, 180.f);
}

// ---- customEnv.py:215-244 -------------------------------------------------------------------------------------
// One command: scale by its bound, clip, report saturation (-1 / 0 / +1).
__device__ __forceinline__ float scale_clip(float a, float bound, int& sat) {
  const float s = __fmul_rn(a, bound);
  sat = (s > bound) - (s < -bound);
  return fminf(fmaxf(s, -bound), bound);
}

// Network action -> clipped real commands cmd[NCMD] (thrust % for bow, port, star, then azimuths).
template <int KIND, bool CONT>
__device__ __forceinline__ void transform_action(const float (&a)[EnvTraits<KIND, CONT>::ACT],
                                                 float (&cmd)[EnvTraits<KIND, CONT>::NCMD],
                                                 int (&sat)[EnvTraits<KIND, CONT>::NCMD]) {
  using T = EnvTraits<KIND, CONT>;
#pragma unroll
  for (int i = 0; i < 3; ++i) cmd[i] = scale_clip(a[i], (float)ML4CA_THRUST_BOUND, sat[i]);
  if constexpr (KIND == ML4CA_ENV_FINAL) {
    if constexpr (CONT) {
      // handle_continuous_angles :227-235 then scale_and_clip: (atan2(s, c) / pi) * pi clipped to +-pi.  The
      // divide/multiply round trip is the identity up to one ulp and |atan2f| <= fl(pi) never clips, so the
      // command is atan2f itself (transcendental piece, tolerance-checked; saves two IEEE divisions per env).
      cmd[3] = fminf(fmaxf(atan2f(a[3], a[4]), -T::ANG_BOUND), T::ANG_BOUND);
      cmd[4] = fminf(fmaxf(atan2f(a[5], a[6]), -T::ANG_BOUND), T::ANG_BOUND);
      sat[3] = sat[4] = 0;
    } else {  // wrap_stern_angles :237-244
      const float ap = __fdiv_rn(wrap_rad(__fmul_rn(a[3], T::ANG_BOUND)), T::ANG_BOUND);
      const float as = __fdiv_rn(wrap_rad(__fmul_rn(a[4], T::ANG_BOUND)), T::ANG_BOUND);
      cmd[3] = scale_clip(ap, T::ANG_BOUND, sat[3]);
      cmd[4] = scale_clip(as, T::ANG_BOUND, sat[4]);
    }
  } else {
#pragma unroll
    for (int i = 3; i < T::NCMD; ++i) cmd[i] = scale_clip(a[i], T::ANG_BOUND, sat[i]);
  }
}

// customEnv.py:117-122: write the azimuth commands into current_angles (env order bow, port, star).
template <int KIND, bool CONT>
__device__ __forceinline__ void apply_angle_commands(const float (&cmd)[EnvTraits<KIND, CONT>::NCMD], float& a_bow,
                                                     float& a_port, float& a_star) {
  if constexpr (KIND == ML4CA_ENV_FULL) {
    a_bow = cmd[3];
    a_port = cmd[4];
    a_star = cmd[5];
  } else if constexpr (KIND == ML4CA_ENV_LIMITED || KIND == ML4CA_ENV_FINAL) {
    a_port = cmd[3];  // act_2_act_map {4:3, 5:4}, customEnv.py:364,392
    a_star = cmd[4];
  }
}

// ---- stand-in hull (DECLARED; see ml4ca_constants.h and oracle/vessel.py) ------------------------------------
__device__ __forceinline__ float fast_sqrt(float x) {  // sqrt.approx: 1 ulp, no IEEE fix-up sequence
  float y;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// (sin, cos) for the hull heading.  |psi| <= pi/4 is the live range of every training env (termination bound
// 45 deg, customEnv.py:386), where the minimax polynomials of the classic single-precision kernels (Cephes sinf /
// cosf, ~1 ulp) need no range reduction: 11 instructions instead of the ~30 of sincosf.  Anything larger takes
// the library route.
__device__ __forceinline__ void sincos_heading(float x, float& s, float& c) {
  if (fabsf(x) <= 0.78539816f) {
    const float z = x * x;
    const float ps = fmaf(fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f), z, -1.6666654611e-1f);
    s = fmaf(ps, z * x, x);
    const float pc = fmaf(fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f), z, 4.166664568298827e-2f);
    c = fmaf(pc, z * z, fmaf(-0.5f, z, 1.0f));
  } else {
    sincosf(x, &s, &c);
  }
}

// x / 100.0f, correctly rounded (== __fdiv_rn(x, 100.0f) bit for bit) in three instructions: q = x * RN(1/100),
// exact remainder r = x - 100 q by FMA, q' = q + r * RN(1/100) (Markstein's correction).  Checked exhaustively
// against IEEE division over every finite float: exact for |x| >= 4.8e-38; the guard routes the denormal
// neighbourhood (and nothing else) to the IEEE sequence.
__device__ __forceinline__ float div100(float x) {
  const float q = __fmul_rn(x, 0.01f);
  const float r = __fmaf_rn(-q, 100.0f, x);
  const float q2 = __fmaf_rn(r, 0.01f, q);
  const bool ok = fabsf(x) >= 1e-30f;
  float res = ok ? q2 : q;                                   // x = +-0 (every freshly reset env): q = +-0 is the quotient
  if (!ok && x != 0.f) res = __fdiv_rn(x, 100.0f);           // denormal neighbourhood only
  return res;
}

// tau = sum_i F_i [cos a_i, sin a_i, lx_i sin a_i - ly_i cos a_i], F_i = K_i n_i |n_i|; env order bow, port, star.
// The caller supplies sin/cos of each azimuth (for the continuous-angle env they come straight from the
// network's (sin, cos) pair: cos(atan2(y, x)) = x / hypot(x, y), no atan2f -> sincosf round trip).
__device__ __forceinline__ void thruster_wrench_sc(float n_bow, float n_port, float n_star, float sb, float cb,
                                                   float sp, float cp, float ss, float cs, float& tx, float& ty,
                                                   float& tn) {
  const float fb = (float)ML4CA_K_BOW * n_bow * fabsf(n_bow);
  const float fp = (float)ML4CA_K_STERN * n_port * fabsf(n_port);
  const float fs = (float)ML4CA_K_STERN * n_star * fabsf(n_star);
  tx = fb * cb + fp * cp + fs * cs;
  ty = fb * sb + fp * sp + fs * ss;
  tn = fb * ((float)ML4CA_LX_BOW * sb - (float)ML4CA_LY_BOW * cb) +
       fp * ((float)ML4CA_LX_PORT * sp - (float)ML4CA_LY_PORT * cp) +
       fs * ((float)ML4CA_LX_STAR * ss - (float)ML4CA_LY_STAR * cs);
}

// (sin, cos) of atan2(y, x) without evaluating the angle: (y, x) / hypot(x, y); atan2(0, 0) = 0 -> (0, 1).
__device__ __forceinline__ void unit_from_pair(float y, float x, float& s, float& c) {
  const float h2 = x * x + y * y;
  const float inv = rsqrtf(h2);
  const bool ok = h2 > 1e-30f && h2 < 1e30f;
  s = ok ? y * inv : 0.f;
  c = ok ? x * inv : 1.f;
  if (!ok && h2 != 0.f) sincosf(atan2f(y, x), &s, &c);  // denormal / overflow corner: exact route
}

// atan2(s, c) of a UNIT vector, branch-free: a = min(|s|, |c|) / max(|s|, |c|) in [0, 1] (the max is >= 0.707, so the
// MUFU reciprocal is safe), odd minimax polynomial of degree 15 (max error 1.2e-7 rad in fp32, the size of one ulp of
// pi), octant / quadrant / sign fix-ups by selects.  ~20 instructions against ~45 with branches for atan2f.
__device__ __forceinline__ float atan2_unit(float s, float c) {
  const float as = fabsf(s), ac = fabsf(c);
  const float mx = fmaxf(as, ac), mn = fminf(as, ac);
  const float a = mn * __frcp_rn(mx);
  const float z = a * a;
  float p = -0.004054387100040913f;
  p = fmaf(p, z, 0.021862266585230827f);
  p = fmaf(p, z, -0.05591126158833504f);
  p = fmaf(p, z, 0.09642113000154495f);
  p = fmaf(p, z, -0.13908593356609344f);
  p = fmaf(p, z, 0.1994655728340149f);
  p = fmaf(p, z, -0.33329859375953674f);
  p = fmaf(p, z, 0.9999993443489075f);
  float r = p * a;
  r = as > ac ? 1.5707963267948966f - r : r;
  r = c < 0.f ? 3.14159265358979323846f - r : r;
  return copysignf(r, s);
}

// RevoltFinal with continuous angles on the step path: thrust commands as in transform_action, azimuth commands and
// their (sin, cos) from the network's pairs without atan2f / sincosf.
__device__ __forceinline__ void transform_action_final_cont(const float (&a)[7], float (&cmd)[5], int (&sat)[5], float& sp,
                                                            float& cp, float& ss, float& cs) {
#pragma unroll
  for (int i = 0; i < 3; ++i) cmd[i] = scale_clip(a[i], (float)ML4CA_THRUST_BOUND, sat[i]);
  unit_from_pair(a[3], a[4], sp, cp);
  unit_from_pair(a[5], a[6], ss, cs);
  cmd[3] = fminf(fmaxf(atan2_unit(sp, cp), -kPi), kPi);     // handle_continuous_angles + scale_and_clip, :227-235,215-225
  cmd[4] = fminf(fmaxf(atan2_unit(ss, cs), -kPi), kPi);
  sat[3] = sat[4] = 0;
}

// Per-launch constants of the integrator, folded on the host (hull_consts()).
struct HullConsts {
  float h;                    // sub-step, s
  float hm1, hm2, hm3;        // h / m11, h / m22, h / m33
  float k_vr, k_ur, k_uv;     // Coriolis couplings times h / m
  float one_xu, xuu, one_yv, yvv, one_nr, nrr;  // 1 - h Xu/m11, h Xuu/m11, ...
  float rot_c2, rot_s1, rot_s3;  // -h^2/2, h, -h^3/6: small-angle rotation kernel in terms of r
  float lag_k;                // h / (T + h): gain of the wrench lag per sub-step (1 = no lag)
};

// `model`: ml4ca_env_cfg.hull_model (0 = default constants, 1 = the box-test fit, ml4ca_constants.h); `lag_s`:
// ml4ca_env_cfg.actuator_lag_s.
inline HullConsts hull_consts(float h, int model = 0, float lag_s = 0.f) {
  const bool fit = model == 1;
  const double m11 = fit ? ML4CA_H1_M11 : ML4CA_M11, m22 = fit ? ML4CA_H1_M22 : ML4CA_M22, m33 = fit ? ML4CA_H1_M33 : ML4CA_M33;
  const double xu = fit ? ML4CA_H1_XU : ML4CA_XU, xuu = fit ? ML4CA_H1_XUU : ML4CA_XUU;
  const double yv = fit ? ML4CA_H1_YV : ML4CA_YV, yvv = fit ? ML4CA_H1_YVV : ML4CA_YVV;
  const double nr = fit ? ML4CA_H1_NR : ML4CA_NR, nrr = fit ? ML4CA_H1_NRR : ML4CA_NRR;
  HullConsts k;
  k.h = h;
  k.hm1 = (float)((double)h / m11);
  k.hm2 = (float)((double)h / m22);
  k.hm3 = (float)((double)h / m33);
  k.k_vr = (float)((double)h * m22 / m11);
  k.k_ur = (float)((double)h * m11 / m22);
  k.k_uv = (float)((double)h * (m22 - m11) / m33);
  k.one_xu = (float)(1.0 - (double)h * xu / m11);
  k.xuu = (float)((double)h * xuu / m11);
  k.one_yv = (float)(1.0 - (double)h * yv / m22);
  k.yvv = (float)((double)h * yvv / m22);
  k.one_nr = (float)(1.0 - (double)h * nr / m33);
  k.nrr = (float)((double)h * nrr / m33);
  k.rot_c2 = (float)(-0.5 * (double)h * h);
  k.rot_s1 = h;
  k.rot_s3 = (float)(-(double)h * h * h / 6.0);
  k.lag_k = lag_s > 0.f ? (float)((double)h / ((double)lag_s + (double)h)) : 1.0f;
  return k;
}

// n_sub semi-implicit Euler sub-steps:  nu+ = nu + h nu_dot(nu);  N,E += h R(psi) nu+;  psi += h r+.
// 25 FP32 instructions per sub-step:
//  * nu+ = (1 - h d(nu)/m) nu + h (tau + coriolis)/m      -- 3 products + 3 x 3 FMA
//  * the pose increments are summed un-scaled (sum R nu, sum r) and multiplied by h once, apart from the pose
//    itself, so 20 small additions do not each round at the magnitude of N, E
//  * R(psi) advances by the angle-sum recurrence with the small-angle kernel (cos, sin)(h r) ~ (1 - (h r)^2 / 2, h r):
//    |h r| <= 5.2e-3, so the heading used for the position increments drifts by (h r)^3 / 6 <= 2.3e-8 rad per
//    sub-step (<= 7e-8 m per env step at top speed, below the fp32 resolution of N, E); (s, c) are re-derived from
//    psi at every env step and psi itself is the exact sum of h r.
__device__ __forceinline__ void integrate_hull(float& N, float& E, float& psi, float& u, float& v, float& r,
                                               float tx, float ty, float tn, int n_sub, const HullConsts& k) {
  const float ax = k.hm1 * tx, ay = k.hm2 * ty, an = k.hm3 * tn;
  float s, c;
  sincos_heading(psi, s, c);
  float sN = 0.f, sE = 0.f, sr = 0.f;
#pragma unroll 5
  for (int i = 0; i < n_sub; ++i) {
    const float vr = v * r, ur = u * r, uv = u * v;
    const float un = fmaf(fmaf(-k.xuu, fabsf(u), k.one_xu), u, fmaf(k.k_vr, vr, ax));
    const float vn = fmaf(fmaf(-k.yvv, fabsf(v), k.one_yv), v, fmaf(-k.k_ur, ur, ay));
    const float rn = fmaf(fmaf(-k.nrr, fabsf(r), k.one_nr), r, fmaf(-k.k_uv, uv, an));
    u = un;
    v = vn;
    r = rn;
    sN = fmaf(-s, v, fmaf(c, u, sN));
    sE = fmaf(c, v, fmaf(s, u, sE));
    sr += r;
    const float r2 = r * r;
    const float cd = fmaf(k.rot_c2, r2, 1.0f);
    const float sd = r * k.rot_s1;
    const float cn = fmaf(-s, sd, c * cd);
    s = fmaf(c, sd, s * cd);
    c = cn;
  }
  N = fmaf(k.h, sN, N);
  E = fmaf(k.h, sE, E);
  psi = fmaf(k.h, sr, psi);
}

// integrate_hull with a first-order lag of the thruster wrench (ml4ca_env_cfg.actuator_lag_s > 0; oracle/vessel.py):
// tau_act is a state of the env; every sub-step first moves it towards the command by lag_k, then advances the hull with it.
// Nine more FP32 instructions per sub-step than integrate_hull.
// FORCE: (fx, fy, fn) is a body-frame force added to the lagged wrench (the environmental bias, which is not lagged).
template <bool FORCE = false>
__device__ __forceinline__ void integrate_hull_lag(float& N, float& E, float& psi, float& u, float& v, float& r,
                                                   float tx, float ty, float tn, float& ta_x, float& ta_y, float& ta_n,
                                                   int n_sub, const HullConsts& k, float fx = 0.f, float fy = 0.f,
                                                   float fn = 0.f) {
  float s, c;
  sincos_heading(psi, s, c);
  float sN = 0.f, sE = 0.f, sr = 0.f;
#pragma unroll 5
  for (int i = 0; i < n_sub; ++i) {
    ta_x = fmaf(k.lag_k, tx - ta_x, ta_x);
    ta_y = fmaf(k.lag_k, ty - ta_y, ta_y);
    ta_n = fmaf(k.lag_k, tn - ta_n, ta_n);
    const float vr = v * r, ur = u * r, uv = u * v;
    const float fx_ = FORCE ? ta_x + fx : ta_x, fy_ = FORCE ? ta_y + fy : ta_y, fn_ = FORCE ? ta_n + fn : ta_n;
    const float un = fmaf(fmaf(-k.xuu, fabsf(u), k.one_xu), u, fmaf(k.k_vr, vr, k.hm1 * fx_));
    const float vn = fmaf(fmaf(-k.yvv, fabsf(v), k.one_yv), v, fmaf(-k.k_ur, ur, k.hm2 * fy_));
    const float rn = fmaf(fmaf(-k.nrr, fabsf(r), k.one_nr), r, fmaf(-k.k_uv, uv, k.hm3 * fn_));
    u = un;
    v = vn;
    r = rn;
    sN = fmaf(-s, v, fmaf(c, u, sN));
    sE = fmaf(c, v, fmaf(s, u, sE));
    sr += r;
    const float r2 = r * r;
    const float cd = fmaf(k.rot_c2, r2, 1.0f);
    const float sd = r * k.rot_s1;
    const float cn = fmaf(-s, sd, c * cd);
    s = fmaf(c, sd, s * cd);
    c = cn;
  }
  N = fmaf(k.h, sN, N);
  E = fmaf(k.h, sE, E);
  psi = fmaf(k.h, sr, psi);
}

// Two environments per thread on the packed FP32 pipe (FFMA2 / FMUL2 / FADD2, sm_100a): the same recurrence as
// integrate_hull, operand for operand (every lane rounds exactly like the scalar code), at 14 issue slots per
// environment sub-step instead of 25.  The damping factors stay scalar FFMAs: |.| is a free operand modifier
// there, while the packed form would need separate abs instructions.
__device__ __forceinline__ float2 splat2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ void integrate_hull2(float2& N, float2& E, float2& psi, float2& u, float2& v, float2& r,
                                                float2 tx, float2 ty, float2 tn, int n_sub, const HullConsts& k) {
  const float2 ax = __fmul2_rn(splat2(k.hm1), tx), ay = __fmul2_rn(splat2(k.hm2), ty), an = __fmul2_rn(splat2(k.hm3), tn);
  float2 s, c;
  sincos_heading(psi.x, s.x, c.x);
  sincos_heading(psi.y, s.y, c.y);
  float2 sN = splat2(0.f), sE = splat2(0.f), sr = splat2(0.f);
  const float2 kvr = splat2(k.k_vr), nkur = splat2(-k.k_ur), nkuv = splat2(-k.k_uv);
  const float2 c2 = splat2(k.rot_c2), s1 = splat2(k.rot_s1), one = splat2(1.0f);
#pragma unroll 5
  for (int i = 0; i < n_sub; ++i) {
    const float2 vr = __fmul2_rn(v, r), ur = __fmul2_rn(u, r), uv = __fmul2_rn(u, v);
    const float2 du = make_float2(fmaf(-k.xuu, fabsf(u.x), k.one_xu), fmaf(-k.xuu, fabsf(u.y), k.one_xu));
    const float2 dv = make_float2(fmaf(-k.yvv, fabsf(v.x), k.one_yv), fmaf(-k.yvv, fabsf(v.y), k.one_yv));
    const float2 dr = make_float2(fmaf(-k.nrr, fabsf(r.x), k.one_nr), fmaf(-k.nrr, fabsf(r.y), k.one_nr));
    u = __ffma2_rn(du, u, __ffma2_rn(kvr, vr, ax));
    v = __ffma2_rn(dv, v, __ffma2_rn(nkur, ur, ay));
    r = __ffma2_rn(dr, r, __ffma2_rn(nkuv, uv, an));
    sN = __ffma2_rn(neg2(s), v, __ffma2_rn(c, u, sN));
    sE = __ffma2_rn(c, v, __ffma2_rn(s, u, sE));
    sr = __fadd2_rn(sr, r);
    const float2 r2 = __fmul2_rn(r, r);
    const float2 cd = __ffma2_rn(c2, r2, one);
    const float2 sd = __fmul2_rn(r, s1);
    const float2 cn = __ffma2_rn(neg2(s), sd, __fmul2_rn(c, cd));
    s = __ffma2_rn(c, sd, __fmul2_rn(s, cd));
    c = cn;
  }
  const float2 h = splat2(k.h);
  N = __ffma2_rn(h, sN, N);
  E = __ffma2_rn(h, sE, E);
  psi = __ffma2_rn(h, sr, psi);
}

// ---- errorFrame.py:25-32 --------------------------------------------------------------------------------------
__device__ __forceinline__ void error_frame(float N, float E, float psi, float rN, float rE, float rpsi, float& xb,
                                            float& yb, float& psib) {
  const float eN = __fsub_rn(N, rN), eE = __fsub_rn(E, rE), ep = __fsub_rn(psi, rpsi);
  float s, c;
  sincos_heading(wrap_deg_quirk(psi), s, c);
  xb = c * eN + s * eE;  // R(psi)^T e
  yb = c * eE - s * eN;
  psib = wrap_deg_quirk(ep);
}

// ---- customEnv.py:253-325, coefficients of :263 -----------------------------------------------------------------
// thrust[3] = this step's clipped thrust (the NEW prev_thrust, :126), old_thrust[3] = the previous step's thrust
// (the reference reads it back as state_ext[-3:] * 100, :311), angle deltas = current_angles - prev_angles, env
// order bow, port, star.  Tolerance-checked piece: quotients by constants are products with the reciprocal,
// sqrt/exp use the MUFU approximations (<= 2 ulp); inv_dt = 1 / step_dt, inv_bound = 1 / real_action_bounds[4].
template <bool EXT>
__device__ __forceinline__ float reward_fn(float xb, float yb, float psib, float u, float v, float r,
                                           const float (&thrust)[3], const float (&old_thrust)[3], float da_bow,
                                           float da_port, float da_star, float inv_dt, float inv_bound) {
  // vel_reward :267-273
  const float vel = -fast_sqrt((u * u) * (float)ML4CA_REW_VEL_CU + (v * v) * (float)ML4CA_REW_VEL_CV +
                               (r * r) * (float)ML4CA_REW_VEL_CR);
  // multivariate_gaussian :275-290
  const float d2 = xb * xb + yb * yb;
  const float yaw = psib * (float)(180.0 / ML4CA_PI);
  const float y2 = yaw * yaw;
  const float quad = d2 * (float)(1.0 / (ML4CA_REW_SIGMA_POS * ML4CA_REW_SIGMA_POS)) +
                     y2 * (float)(1.0 / (ML4CA_REW_SIGMA_YAW * ML4CA_REW_SIGMA_YAW));
  const float multivar = 2.0f * __expf(-0.5f * quad);
  const float special = fast_sqrt(fmaf(y2, 0.0625f, d2));
  const float anti = fmaxf(-1.0f, fmaf(-0.1f, special, 1.0f));
  float rew = vel + (multivar + anti + 0.5f);
  // thrust_penalty :292-302
  rew -= fabsf(thrust[0]) * (float)(ML4CA_REW_THRUST_C_BOW / 100.0);
  rew -= (fabsf(thrust[1]) + fabsf(thrust[2])) * (float)(ML4CA_REW_THRUST_C_STERN / 100.0);
  // action_derivative_penalty :304-325 (returns 0 without the extended state)
  if constexpr (EXT) {
    const float kd = inv_dt * (float)(ML4CA_REW_DTHRUST_C / 100.0);
    const float pen = (fabsf(thrust[0] - old_thrust[0]) + fabsf(thrust[1] - old_thrust[1]) +
                       fabsf(thrust[2] - old_thrust[2])) * kd;
    const float ka = inv_dt * inv_bound;
    const float angpen = fabsf(da_bow) * (ka * (float)ML4CA_REW_DANGLE_C_BOW) +
                         (fabsf(da_port) + fabsf(da_star)) * (ka * (float)ML4CA_REW_DANGLE_C_STERN);
    rew -= pen + fminf(1.0f, angpen);
  }
  return rew;
}

// customEnv.py:207-213: any(|obs[i]| > bound[i]), i < 6, strict.
__device__ __forceinline__ bool is_terminal(float xb, float yb, float psib, float u, float v, float r,
                                            const float* __restrict__ b) {
  return (fabsf(xb) > b[0]) | (fabsf(yb) > b[1]) | (fabsf(psib) > b[2]) | (fabsf(u) > b[3]) | (fabsf(v) > b[4]) |
         (fabsf(r) > b[5]);
}

// Episode word: one int32 per env = (episode counter mod 2^16) << 16 | steps taken in the current episode.
// One row instead of two keeps the in-kernel restart free of a dependent load: the word is on the step path
// anyway (episode-length cut, ppo.py:304).  The Philox counter of a restart is the word at that moment, so
// the draws of an env repeat only if episode number (mod 65536) AND episode length coincide.
constexpr uint32_t kEpLenMask = 0xFFFFu;
__device__ __forceinline__ int32_t next_episode_word(int32_t w) { return (int32_t)((((uint32_t)w >> 16) + 1u) << 16); }

// customEnv.py:141-145 + simtools.py:109-124 on the Philox stream: pose ~ U(+-fraction*b[0:3]),
// velocity ~ U(+-0.30*fraction*b[3:6]).  scale[6] is precomputed on the host in fp32 (see make_reset_scale).
// `episode` is the env's episode word at the moment of the reset.
__device__ __forceinline__ void sample_reset(uint64_t seed, int64_t env_id, int32_t episode,
                                             const float* __restrict__ scale, float& N, float& E, float& psi, float& u,
                                             float& v, float& r) {
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ 0x5EED5EEDu;
  const uint32_t lo = (uint32_t)((uint64_t)env_id), hi = (uint32_t)((uint64_t)env_id >> 32);
  // one Philox block = 128 bits = six 21-bit uniforms (resolution 2^-20 of each interval)
  const Philox4 q = philox4x32_10(lo, hi, (uint32_t)episode, kTagResetPose, k0, k1);
  N = __fmul_rn(scale[0], symmetric_unit21(q.x));
  E = __fmul_rn(scale[1], symmetric_unit21(q.y));
  psi = __fmul_rn(scale[2], symmetric_unit21(q.z));
  u = __fmul_rn(scale[3], symmetric_unit21(q.w));
  v = __fmul_rn(scale[4], symmetric_unit21(((q.x >> 21) | (q.y >> 21 << 11)) & 0x1FFFFFu));
  r = __fmul_rn(scale[5], symmetric_unit21(((q.z >> 21) | (q.w >> 21 << 11)) & 0x1FFFFFu));
}

// Three standard normals from one Philox block of (env, episode word, tag): Box-Muller on (x, y) -> r0 cos, r0 sin and
// on (z, w) -> r1 cos, with r = sqrt(-2 ln unit_open(.)), angle = 2 pi (. >> 8) 2^-24 (tests/disturbance_oracle.py::normals3).
__device__ __forceinline__ void philox_normals3(uint64_t seed, int64_t env_id, int32_t episode, uint32_t tag,
                                                float (&z)[3]) {
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ 0x5EED5EEDu;
  const uint32_t lo = (uint32_t)((uint64_t)env_id), hi = (uint32_t)((uint64_t)env_id >> 32);
  const Philox4 q = philox4x32_10(lo, hi, (uint32_t)episode, tag, k0, k1);
  const float r0 = sqrtf(-2.0f * logf(unit_open(q.x))), r1 = sqrtf(-2.0f * logf(unit_open(q.z)));
  float s0, c0, s1, c1;
  sincospif((float)(q.y >> 8) * 1.1920928955078125e-07f, &s0, &c0);   // angle = 2 pi * (y >> 8) * 2^-24
  sincospif((float)(q.w >> 8) * 1.1920928955078125e-07f, &s1, &c1);
  z[0] = r0 * c0, z[1] = r0 * s0, z[2] = r1 * c1;
}

// customEnv.py:179-188 (reset_acts=True): prev_thrust <- scale_and_clip([N(0, 0.1)]^3) = clip(100 * (0.1 z), +-100);
// the thrust commands themselves only reach the simulator after the settle steps and are overwritten by the next
// step's action, so the previous-thrust state (observation tail + first derivative penalty) is the whole effect.
// Second Philox block of the restart (counter word 3 = 1), Box-Muller on (x, y) and (z, w).  Rare path: kept out
// of line so that logf / sincospif do not enter the step kernel's register budget.
static __device__ __noinline__ void sample_reset_thrust(uint64_t seed, int64_t env_id, int32_t episode, float* __restrict__ t) {
  float z[3];
  philox_normals3(seed, env_id, episode, kTagResetThrust, z);
#pragma unroll
  for (int c = 0; c < 3; ++c) t[c] = fminf(fmaxf(__fmul_rn(__fmul_rn(0.1f, z[c]), 100.0f), -100.0f), 100.0f);
}

// ---- environmental disturbance (DECLARED model, DESIGN.md section 4; tests/disturbance_oracle.py) ------------------------------
// Ocean current v_c = V [cos beta, sin beta] (NED, constant over an episode) and a NED bias force b = [X_N, Y_E, N_psi]
// following the first-order Gauss-Markov process b <- a b + sigma sqrt(1 - a^2) w per env step, a = exp(-step_dt / T_b)
// (T_b = 0: a = 1, constant over the episode).  Per-launch constants, folded on the host (ml4ca_env_set_disturbance).
struct DistConsts {
  float speed_lo, speed_span;   // V ~ U(speed_lo, speed_lo + speed_span), m/s
  float dir_lo, dir_span;       // beta ~ U(dir_lo, dir_lo + dir_span), rad: the direction the water flows towards
  float bias_std[3];            // sigma: stationary std of b (N, N, Nm); a reset draws b = sigma w0
  float gm_a;                   // a
  float gm_gain[3];             // sigma sqrt(1 - a^2)
  float t_step;                 // n_sub * h: time one env step integrates (drift of the pose with the current)
  int32_t gm;                   // 1: b is updated every env step (T_b > 0)
  int32_t noise;                // 1: ... with a random term (some sigma > 0); 0: b <- a b only
};

// Uniform in [0, 1) from the top 24 bits: (x >> 8) * 2^-24, exact in fp32.
__device__ __forceinline__ float unit01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }

// Current of a new episode: third Philox block of the restart (counter word 3 = kTagCurrent); speed from x, direction
// from y.  `episode` is the episode word at the moment of the reset, as for sample_reset.
__device__ __forceinline__ void sample_current(uint64_t seed, int64_t env_id, int32_t episode, const DistConsts& d,
                                               float& cN, float& cE) {
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ 0x5EED5EEDu;
  const uint32_t lo = (uint32_t)((uint64_t)env_id), hi = (uint32_t)((uint64_t)env_id >> 32);
  const Philox4 q = philox4x32_10(lo, hi, (uint32_t)episode, kTagCurrent, k0, k1);
  const float V = fmaf(d.speed_span, unit01(q.x), d.speed_lo);
  const float beta = fmaf(d.dir_span, unit01(q.y), d.dir_lo);
  float s, c;
  sincosf(beta, &s, &c);
  cN = V * c;
  cE = V * s;
}

// The disturbance state of a new episode: the current and b = sigma w0 (stationary draw, counter word 3 = kTagBias0).
// Rare path (resets only), kept out of line like sample_reset_thrust.
static __device__ __noinline__ void sample_disturbance(uint64_t seed, int64_t env_id, int32_t episode, const DistConsts& d,
                                                       float* __restrict__ cur, float* __restrict__ b) {
  sample_current(seed, env_id, episode, d, cur[0], cur[1]);
  float z[3];
  philox_normals3(seed, env_id, episode, kTagBias0, z);
#pragma unroll
  for (int c = 0; c < 3; ++c) b[c] = d.bias_std[c] * z[c];
}

// One env step of the Gauss-Markov bias.  `word` is the episode word AFTER the step's increment (counter word 3 =
// kTagBiasStep): every step of every episode has its own block, so a replayed CUDA graph draws fresh noise.
__device__ __forceinline__ void advance_bias(uint64_t seed, int64_t env_id, int32_t word, const DistConsts& d,
                                             float& bN, float& bE, float& bP) {
  float z[3] = {0.f, 0.f, 0.f};
  if (d.noise) philox_normals3(seed, env_id, word, kTagBiasStep, z);
  bN = fmaf(d.gm_gain[0], z[0], d.gm_a * bN);
  bE = fmaf(d.gm_gain[1], z[1], d.gm_a * bE);
  bP = fmaf(d.gm_gain[2], z[2], d.gm_a * bP);
}

// ---- first-order wave-frequency motion (DECLARED model, DESIGN.md section 4; tests/wave_oracle.py) ----------------------
// Per env and DOF d (surge, sway, yaw; body frame) the linear oscillator x'' + 2 lambda w0 x' + w0^2 x = sigma_d
// sqrt(4 lambda w0^3) w(t), stationary law P = diag(sigma^2, w0^2 sigma^2).  w0 ~ U(omega range) per episode, shared by
// the three DOFs.  It never feeds back into the hull: it is added to the measured pose and velocity only.
// Per-launch constants, folded on the host (ml4ca_env_set_waves).
struct WaveConsts {
  float sigma[3];               // stationary std of x: m, m, rad
  float omega_lo, omega_span;   // w0 ~ U(omega_lo, omega_lo + omega_span), rad/s
  float lam_dt;                 // lambda * step_dt
  float wd_dt;                  // sqrt(1 - lambda^2) * step_dt: the damped frequency per unit w0, times the step
  float lam_ratio;              // lambda / sqrt(1 - lambda^2)
  float inv_sq;                 // 1 / sqrt(1 - lambda^2)
  int32_t noise;                // 1: some sigma > 0 (the per-step draws run); 0: they are skipped
};

// The wave state of a new episode: w0 from out0 of the kTagWaveOmega block, then the stationary draw x = sigma z1
// (kTagWaveMotion0), x' = w0 sigma z2 (kTagWaveRate0).  `episode` is the episode word at the moment of the reset.  Rare
// path (resets only), kept out of line like sample_disturbance.  The constants come as scalars: a reference into the
// kernel's parameters would make every thread copy them to local memory on entry.
static __device__ __noinline__ void sample_waves(uint64_t seed, int64_t env_id, int32_t episode, float sigma0, float sigma1,
                                                 float sigma2, float omega_lo, float omega_span, float* __restrict__ x,
                                                 float* __restrict__ xd, float* __restrict__ w0) {
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ 0x5EED5EEDu;
  const uint32_t lo = (uint32_t)((uint64_t)env_id), hi = (uint32_t)((uint64_t)env_id >> 32);
  const Philox4 q = philox4x32_10(lo, hi, (uint32_t)episode, kTagWaveOmega, k0, k1);
  const float w = fmaf(omega_span, unit01(q.x), omega_lo);
  const float sigma[3] = {sigma0, sigma1, sigma2};
  float z1[3], z2[3];
  philox_normals3(seed, env_id, episode, kTagWaveMotion0, z1);
  philox_normals3(seed, env_id, episode, kTagWaveRate0, z2);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    x[c] = sigma[c] * z1[c];
    xd[c] = w * (sigma[c] * z2[c]);
  }
  *w0 = w;
}

// One env step of the wave motion, the exact discretisation s <- Phi s + sigma L z of s = [x, x'] over step_dt.  In the
// scaled state y = x' / w0 the stationary covariance is the identity, so Phi' = D^-1 Phi D (D = diag(1, w0)) with
//   e = exp(-lambda w0 dt), (sn, cs) = (sin, cos)(w0 sqrt(1 - lambda^2) dt), g = e sn / sqrt(1 - lambda^2):
//   Phi' = [[e (cs + lambda' sn), g], [-g, e (cs - lambda' sn)]],  lambda' = lambda / sqrt(1 - lambda^2),
// Q' = I - Phi' Phi'^T and L' its Cholesky factor (L = D L').  The diagonal of Q' is O((w0 dt)^3) small; written as
// Q'11 = (1 - e^2) - 2 lambda' sn e Phi'11 and Q'22 = (1 - e^2) + 2 lambda' sn e Phi'22 (with 1 - e^2 from expm1f) it does
// not cancel against 1 in fp32.  `word` is the episode word AFTER the step's increment: the two normals of each DOF come
// from the kTagWaveStep1 / kTagWaveStep2 blocks of it.
__device__ __forceinline__ void advance_waves(uint64_t seed, int64_t env_id, int32_t word, const WaveConsts& k, float w0,
                                              float (&x)[3], float (&xd)[3]) {
  const float e = expf(-k.lam_dt * w0);
  float sn, cs;
  sincosf(k.wd_dt * w0, &sn, &cs);
  const float g = e * sn * k.inv_sq;
  const float f11 = e * fmaf(k.lam_ratio, sn, cs), f22 = e * fmaf(-k.lam_ratio, sn, cs);
  const float one_m_e2 = -expm1f(-2.0f * k.lam_dt * w0), h = 2.0f * k.lam_ratio * sn * e;
  const float q11 = fmaf(-h, f11, one_m_e2), q22 = fmaf(h, f22, one_m_e2), q12 = g * (f11 - f22);
  const float l11 = sqrtf(fmaxf(q11, 0.f));
  const float l21 = l11 > 0.f ? q12 / l11 : 0.f;
  const float l22 = sqrtf(fmaxf(fmaf(-l21, l21, q22), 0.f));
  float z1[3] = {0.f, 0.f, 0.f}, z2[3] = {0.f, 0.f, 0.f};
  if (k.noise) {
    philox_normals3(seed, env_id, word, kTagWaveStep1, z1);
    philox_normals3(seed, env_id, word, kTagWaveStep2, z2);
  }
  const float iw = 1.0f / w0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float y = xd[c] * iw;
    const float xn = fmaf(f11, x[c], fmaf(g, y, k.sigma[c] * (l11 * z1[c])));
    const float yn = fmaf(-g, x[c], fmaf(f22, y, k.sigma[c] * fmaf(l21, z1[c], l22 * z2[c])));
    x[c] = xn;
    xd[c] = w0 * yn;
  }
}

// The measured pose and velocity: the LF pose plus the wave motion rotated by the LF heading psi (x_s surge, x_w sway),
// psi + x_psi, and nu + x' (body frame).  In place.
__device__ __forceinline__ void add_wave_motion(float& N, float& E, float& psi, float& u, float& v, float& r,
                                                const float (&x)[3], const float (&xd)[3]) {
  float s, c;
  sincos_heading(psi, s, c);
  N = fmaf(c, x[0], fmaf(-s, x[1], N));
  E = fmaf(s, x[0], fmaf(c, x[1], E));
  psi += x[2];
  u += xd[0], v += xd[1], r += xd[2];
}

}  // namespace ml4ca
