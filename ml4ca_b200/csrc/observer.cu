// observer.cu -- passive nonlinear DP observer (Fossen & Strand, Automatica 35 (1999); Fossen, Handbook of Marine Craft
// Hydrodynamics and Motion Control (2011) section 11.4.1), one thread per environment.
//
// ABSENT FROM THE REFERENCE like the PID (DNV GL's dp_controller stack, qp_allocator.py:6,83): the equations below are
// this build's own statement (DESIGN.md section 4, "DP observer"); tests/observer_oracle.py restates the discrete
// recurrence in float64.
//
//   y~     = y - eta^ - xi2^                       (yaw component wrapped to [-pi, pi); eta^_psi is not wrapped)
//   xi1^'  = xi2^ + K11 y~                         wave model  eta_w = xi2,  s / (s^2 + 2 lambda w_o s + w_o^2) per DOF
//   xi2^'  = -w_o^2 xi1^ - 2 lambda w_o xi2^ + K12 y~
//   eta^'  = R(psi_m) nu^ + K2 y~
//   b^'    = -b^ / T_b + K3 y~                     (T_b = 0: no decay)
//   M nu^' = tau - D(nu^) nu^ - Coriolis(nu^) + R(psi_m)^T (b^ + K4 y~)
//
// M, D and the Coriolis couplings are the env's declared hull (hull_consts() of env_math.cuh, no second copy); tau is
// thruster_wrench_sc of the thrust and azimuths the env step just applied; psi_m is the measured heading, held over
// the step.  K11 = -2 (zeta_n - lambda) w_c / w_o, K12 = 2 w_o (zeta_n - lambda), K2 = w_c = cutoff_ratio w_o per DOF.
//
// Discretisation: y, tau and psi_m are held over the env step (zero-order hold); n_sub = max(1, round(step_dt / sim_dt))
// semi-implicit Euler sub-steps of h = step_dt / n_sub, with y~ recomputed every sub-step: the velocity-type states
// (xi2^, nu^, b^) advance from the old state first, then the position-type states (xi1^, eta^) with the new xi2^, nu^.
//
// State: one caller-owned [15, n] fp32 tensor, rows xi1^[3], xi2^[3], eta^[3] (N, E, psi), nu^[3] (u, v, r), b^[3] (NED:
// N, N, Nm, the frame and units of the env's bias).  161 algorithmic bytes per env-step: read state 60, y 12, thrust 12,
// angles 12, w_o 4, restart 1; write state 60.
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

__global__ void __launch_bounds__(256) observer_step_kernel(int64_t n, const ObsConsts k, const float* __restrict__ y_,
                                                            const float* __restrict__ thrust, const float* __restrict__ angles,
                                                            const float* __restrict__ omega, const uint8_t* __restrict__ restart,
                                                            float* __restrict__ state) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float x[15], y[3], th[3], an[3];
#pragma unroll
  for (int r = 0; r < 15; ++r) x[r] = state[(int64_t)r * n + i];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    y[c] = y_[(int64_t)c * n + i];
    th[c] = thrust[(int64_t)c * n + i];
    an[c] = angles[(int64_t)c * n + i];
  }
  const float w = clamp_omega(omega[i]);
  const bool again = restart != nullptr && restart[i] != 0;
  if (again) {
    observer_reset_column(x, y);
  } else {
    float sb, cb, sp, cp, ss, cs;
    sincosf(an[0], &sb, &cb);
    sincosf(an[1], &sp, &cp);
    sincosf(an[2], &ss, &cs);
    float tx, ty, tn;
    thruster_wrench_sc(th[0], th[1], th[2], sb, cb, sp, cp, ss, cs, tx, ty, tn);
    observer_advance(x, y, tx, ty, tn, w, k);
  }
#pragma unroll
  for (int r = 0; r < 15; ++r) state[(int64_t)r * n + i] = x[r];
}

__global__ void __launch_bounds__(256) observer_reset_kernel(int64_t n, const float* __restrict__ y_,
                                                             const uint8_t* __restrict__ mask, float* __restrict__ state) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (mask != nullptr && mask[i] == 0) return;
  float x[15];
  const float y[3] = {y_[i], y_[n + i], y_[2 * n + i]};
  observer_reset_column(x, y);
#pragma unroll
  for (int r = 0; r < 15; ++r) state[(int64_t)r * n + i] = x[r];
}

static int validate_observer_cfg(const ml4ca_observer_cfg* c) {
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

static ObsConsts observer_consts(const ml4ca_observer_cfg& c) {
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

using namespace ml4ca;

extern "C" {

int ml4ca_observer_cfg_default(int32_t hull_model, ml4ca_observer_cfg* cfg) {
  ML4CA_REQUIRE(cfg != nullptr, "cfg is NULL");
  ML4CA_REQUIRE(hull_model == 0 || hull_model == 1, "hull_model must be 0 or 1");
  const bool fit = hull_model == 1;
  const double m[3] = {fit ? ML4CA_H1_M11 : ML4CA_M11, fit ? ML4CA_H1_M22 : ML4CA_M22, fit ? ML4CA_H1_M33 : ML4CA_M33};
  cfg->hull_model = hull_model;
  cfg->step_dt = (float)(ML4CA_N_SUBSTEPS * ML4CA_SIM_DT);
  cfg->notch_damping = (float)ML4CA_OBS_NOTCH_DAMPING;
  cfg->wave_damping = (float)ML4CA_OBS_WAVE_DAMPING;
  cfg->cutoff_ratio = (float)ML4CA_OBS_CUTOFF_RATIO;
  cfg->bias_time_s = (float)ML4CA_OBS_BIAS_TIME_S;
  for (int d = 0; d < 3; ++d) {
    const double k4 = ML4CA_OBS_K4_PER_MASS * m[d];
    cfg->k4[d] = (float)k4;
    cfg->k3[d] = (float)(ML4CA_OBS_K3_PER_K4 * k4);
  }
  return ML4CA_OK;
}

int ml4ca_observer_reset(int64_t n, const float* y, const uint8_t* mask, float* state, void* stream) {
  ML4CA_REQUIRE(n >= 0 && y && state, "n >= 0, y and state are required");
  if (n == 0) return ML4CA_OK;
  observer_reset_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, y, mask, state);
  return check_launch("observer_reset_kernel");
}

int ml4ca_observer_step(const ml4ca_observer_cfg* cfg, int64_t n, const float* y, const float* thrust, const float* angles,
                        const float* omega_o, const uint8_t* restart, float* state, void* stream) {
  const int stv = validate_observer_cfg(cfg);
  if (stv != ML4CA_OK) return stv;
  ML4CA_REQUIRE(n >= 0 && y && thrust && angles && omega_o && state, "n >= 0, y, thrust, angles, omega_o and state are required");
  if (n == 0) return ML4CA_OK;
  const ObsConsts k = observer_consts(*cfg);
  observer_step_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, k, y, thrust, angles,
                                                                                                  omega_o, restart, state);
  return check_launch("observer_step_kernel");
}

}  // extern "C"
