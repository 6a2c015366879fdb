// refmodel.cu -- DP reference model (guidance): a third-order reference filter with saturating elements per env and per
// DOF (Fossen, Handbook of Marine Craft Hydrodynamics and Motion Control (2011) section 12.1), one thread per env.
//
// ABSENT FROM THE REFERENCE like the PID and the observer (DNV GL's dp_controller stack): the model below is this build's
// own statement (DESIGN.md section 4, "DP reference model"); tests/refmodel_oracle.py restates the recurrence in float64.
//
//   eta_d / r = w^3 / ((s + w)(s^2 + 2 zeta w s + w^2))              per DOF N, E, psi (NED)
//   jerk      = w^3 e - (2 zeta + 1) w a_d - (2 zeta + 1) w^2 v_d,   e = r - eta_d   (heading: e wrapped to [-pi, pi))
//
// Discretisation: r held over the env step; n_sub = max(1, round(step_dt / sim_dt)) semi-implicit Euler sub-steps of
// h = step_dt / n_sub, each  a_d <- clamp(a_d + h jerk, +-a_max),  v_d <- clamp(v_d + h a_d, +-v_max),
// eta_d <- eta_d + h v_d.  eta_d,psi is not wrapped (it stays continuous with the vessel heading, as the observer's eta^).
//
// State: one caller-owned [9, n] fp32 tensor, rows eta_d[3], v_d[3], a_d[3].  84 algorithmic bytes per env-step: read
// state 36, set-point 12; write state 36.
#include "refmodel_math.cuh"

namespace ml4ca {

// One thread per env.  A two-envs-per-thread form with 64-bit row accesses (as pinv_pid_kernel<2>) measured 14 % slower
// on a B200 at 16 Mi envs (0.469 against 0.411 ms per step, profiles/refmodel_r3.md); the kernel is issue-bound (53 % of
// the HBM roofline), and the two-env form needed 48 registers against 38.
__global__ void __launch_bounds__(256) refmodel_step_kernel(int64_t n, const RefConsts k, const float* __restrict__ setpoint,
                                                            float* __restrict__ state) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float x[9], r[3];
#pragma unroll
  for (int q = 0; q < 9; ++q) x[q] = state[(int64_t)q * n + i];
#pragma unroll
  for (int d = 0; d < 3; ++d) r[d] = setpoint[(int64_t)d * n + i];
  refmodel_advance(x, r, k);
#pragma unroll
  for (int q = 0; q < 9; ++q) state[(int64_t)q * n + i] = x[q];
}

__global__ void __launch_bounds__(256) refmodel_reset_kernel(int64_t n, const float* __restrict__ eta0,
                                                             float* __restrict__ state) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
#pragma unroll
  for (int d = 0; d < 3; ++d) state[(int64_t)d * n + i] = eta0[(int64_t)d * n + i];
#pragma unroll
  for (int q = 3; q < 9; ++q) state[(int64_t)q * n + i] = 0.f;
}

}  // namespace ml4ca

using namespace ml4ca;

extern "C" {

int ml4ca_refmodel_cfg_default(ml4ca_refmodel_cfg* cfg) {
  ML4CA_REQUIRE(cfg != nullptr, "cfg is NULL");
  cfg->step_dt = (float)(ML4CA_N_SUBSTEPS * ML4CA_SIM_DT);
  const double z[3] = {ML4CA_REF_ZETA_N, ML4CA_REF_ZETA_E, ML4CA_REF_ZETA_PSI};
  const double w[3] = {ML4CA_REF_OMEGA_N, ML4CA_REF_OMEGA_E, ML4CA_REF_OMEGA_PSI};
  const double v[3] = {ML4CA_REF_V_MAX_N, ML4CA_REF_V_MAX_E, ML4CA_REF_V_MAX_PSI};
  const double a[3] = {ML4CA_REF_A_MAX_N, ML4CA_REF_A_MAX_E, ML4CA_REF_A_MAX_PSI};
  for (int d = 0; d < 3; ++d) {
    cfg->zeta[d] = (float)z[d];
    cfg->omega[d] = (float)w[d];
    cfg->v_max[d] = (float)v[d];
    cfg->a_max[d] = (float)a[d];
  }
  return ML4CA_OK;
}

int ml4ca_refmodel_reset(int64_t n, const float* eta0, float* state, void* stream) {
  ML4CA_REQUIRE(n >= 0 && eta0 && state, "n >= 0, eta0 and state are required");
  if (n == 0) return ML4CA_OK;
  refmodel_reset_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, eta0, state);
  return check_launch("refmodel_reset_kernel");
}

int ml4ca_refmodel_step(const ml4ca_refmodel_cfg* cfg, int64_t n, const float* setpoint, float* state, void* stream) {
  RefConsts k;
  const int st = refmodel_consts(cfg, k);
  if (st != ML4CA_OK) return st;
  ML4CA_REQUIRE(n >= 0 && setpoint && state, "n >= 0, setpoint and state are required");
  if (n == 0) return ML4CA_OK;
  refmodel_step_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, k, setpoint, state);
  return check_launch("refmodel_step_kernel");
}

}  // extern "C"
