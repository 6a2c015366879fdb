// observer_math.cuh -- the passive DP observer's per-env recurrence (observer.cu states the model) and its host-side
// configuration, shared by the stand-alone observer kernels (observer.cu) and the env-step variant that runs the
// observer in the loop (env_kernels.cuh, OBSV = true).
#pragma once
#include <math.h>

#include "common.h"
#include "env_math.cuh"

namespace ml4ca {

// Per-launch constants, folded on the host from ml4ca_observer_cfg.
struct ObsConsts {
  HullConsts hull;   // h = step_dt / n_sub and the hull terms of the selected model
  int32_t n_sub;
  float hk11;        // h K11 = -2 h (zeta_n - lambda) cutoff_ratio (the same for every DOF and every w_o)
  float two_zl;      // 2 (zeta_n - lambda): K12 = two_zl w_o
  float two_lam;     // 2 lambda
  float cutoff;      // w_c / w_o: K2 = cutoff w_o
  float b_keep;      // 1 - h / T_b (1 when T_b = 0)
  float hk3[3];      // h K3
  float k4[3];       // K4
};

constexpr float kTwoPi = (float)(2.0 * ML4CA_PI);
constexpr float kInvTwoPi = (float)(1.0 / (2.0 * ML4CA_PI));

// a - 2 pi floor((a + pi) / (2 pi)): [-pi, pi) up to the rounding of the product (tests/observer_oracle.py::wrap).
__device__ __forceinline__ float wrap_pi(float a) { return fmaf(-kTwoPi, floorf((a + kPi) * kInvTwoPi), a); }

// One env step of the observer from the held measurement (y, psi_m = y[2]) and body-frame thrust wrench (tx, ty, tn).
// x[15] in the row order of the state tensor, updated in place.
__device__ __forceinline__ void observer_advance(float (&x)[15], const float (&y)[3], float tx, float ty, float tn, float w,
                                                 const ObsConsts& k) {
  const HullConsts& hc = k.hull;
  const float h = hc.h;
  float s, c;
  sincosf(y[2], &s, &c);
  const float hw2 = h * (w * w);                       // h w_o^2
  const float damp = fmaf(-h * k.two_lam, w, 1.0f);    // 1 - 2 h lambda w_o
  const float hk12 = h * (k.two_zl * w);               // h K12
  const float hk2 = h * (k.cutoff * w);                // h K2
  const float ax = hc.hm1 * tx, ay = hc.hm2 * ty, an = hc.hm3 * tn;
  float* xi1 = x;
  float* xi2 = x + 3;
  float* eta = x + 6;
  float* nu = x + 9;
  float* b = x + 12;
#pragma unroll 2
  for (int it = 0; it < k.n_sub; ++it) {
    float e[3];
    e[0] = y[0] - eta[0] - xi2[0];
    e[1] = y[1] - eta[1] - xi2[1];
    e[2] = wrap_pi(y[2] - eta[2] - xi2[2]);
    // velocity-type states from the old state
    float x2n[3], g[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      x2n[d] = fmaf(damp, xi2[d], fmaf(-hw2, xi1[d], hk12 * e[d]));
      g[d] = fmaf(k.k4[d], e[d], b[d]);                // b^ + K4 y~ (NED)
    }
    const float fx = fmaf(c, g[0], s * g[1]);          // R(psi_m)^T (b^ + K4 y~)
    const float fy = fmaf(c, g[1], -s * g[0]);
    const float u = nu[0], v = nu[1], r = nu[2];
    const float un = fmaf(fmaf(-hc.xuu, fabsf(u), hc.one_xu), u, fmaf(hc.k_vr, v * r, fmaf(hc.hm1, fx, ax)));
    const float vn = fmaf(fmaf(-hc.yvv, fabsf(v), hc.one_yv), v, fmaf(-hc.k_ur, u * r, fmaf(hc.hm2, fy, ay)));
    const float rn = fmaf(fmaf(-hc.nrr, fabsf(r), hc.one_nr), r, fmaf(-hc.k_uv, u * v, fmaf(hc.hm3, g[2], an)));
#pragma unroll
    for (int d = 0; d < 3; ++d) b[d] = fmaf(k.b_keep, b[d], k.hk3[d] * e[d]);
    nu[0] = un, nu[1] = vn, nu[2] = rn;
    // position-type states with the new xi2^, nu^
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      xi2[d] = x2n[d];
      xi1[d] = fmaf(h, x2n[d], fmaf(k.hk11, e[d], xi1[d]));
    }
    eta[0] = fmaf(h, fmaf(c, un, -s * vn), fmaf(hk2, e[0], eta[0]));
    eta[1] = fmaf(h, fmaf(s, un, c * vn), fmaf(hk2, e[1], eta[1]));
    eta[2] = fmaf(h, rn, fmaf(hk2, e[2], eta[2]));
  }
}

__device__ __forceinline__ void observer_reset_column(float (&x)[15], const float (&y)[3]) {
#pragma unroll
  for (int r = 0; r < 15; ++r) x[r] = 0.f;
  x[6] = y[0], x[7] = y[1], x[8] = y[2];
}

// w_o outside [ML4CA_OBS_OMEGA_MIN, ML4CA_OBS_OMEGA_MAX] is clamped into it; NaN maps to the lower bound (fmaxf returns
// the non-NaN operand).  The row cannot be checked on the host without a copy.
__device__ __forceinline__ float clamp_omega(float w) {
  return fminf(fmaxf(w, (float)ML4CA_OBS_OMEGA_MIN), (float)ML4CA_OBS_OMEGA_MAX);
}

static inline int validate_observer_cfg(const ml4ca_observer_cfg* c) {
  ML4CA_REQUIRE(c != nullptr, "cfg is NULL");
  ML4CA_REQUIRE(c->hull_model == 0 || c->hull_model == 1, "hull_model must be 0 or 1");
  const float v[] = {c->step_dt, c->notch_damping, c->wave_damping, c->cutoff_ratio, c->bias_time_s,
                     c->k3[0], c->k3[1], c->k3[2], c->k4[0], c->k4[1], c->k4[2]};
  for (float x : v) ML4CA_REQUIRE(isfinite(x), "every configuration value must be finite");
  ML4CA_REQUIRE(c->step_dt > 0.f, "step_dt must be > 0");
  ML4CA_REQUIRE(c->wave_damping > 0.f && c->wave_damping < 1.f, "wave_damping (lambda) must lie in (0, 1)");
  ML4CA_REQUIRE(c->notch_damping > c->wave_damping, "notch_damping (zeta_n) must exceed wave_damping (lambda)");
  ML4CA_REQUIRE(c->cutoff_ratio > 1.f, "cutoff_ratio (w_c / w_o) must be > 1");
  ML4CA_REQUIRE(c->bias_time_s >= 0.f, "bias_time_s must be >= 0 (0 = infinity)");
  for (int d = 0; d < 3; ++d) ML4CA_REQUIRE(c->k3[d] >= 0.f && c->k4[d] >= 0.f, "gains k3, k4 must be >= 0");
  return ML4CA_OK;
}

static inline ObsConsts observer_consts(const ml4ca_observer_cfg& c) {
  const double dt = c.step_dt;
  const int n_sub = (int)fmax(1.0, nearbyint(dt / ML4CA_SIM_DT));
  const float h = (float)(dt / n_sub);
  ObsConsts k;
  k.hull = hull_consts(h, c.hull_model);
  k.n_sub = n_sub;
  const double zl = (double)c.notch_damping - (double)c.wave_damping;
  k.hk11 = (float)(-2.0 * (double)h * zl * c.cutoff_ratio);
  k.two_zl = (float)(2.0 * zl);
  k.two_lam = (float)(2.0 * c.wave_damping);
  k.cutoff = c.cutoff_ratio;
  k.b_keep = c.bias_time_s > 0.f ? (float)(1.0 - (double)h / c.bias_time_s) : 1.0f;
  for (int d = 0; d < 3; ++d) {
    k.hk3[d] = (float)((double)h * c.k3[d]);
    k.k4[d] = c.k4[d];
  }
  return k;
}

}  // namespace ml4ca
