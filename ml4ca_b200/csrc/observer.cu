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
#include "observer_math.cuh"

namespace ml4ca {

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
