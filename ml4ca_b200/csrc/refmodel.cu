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
#include "observer_math.cuh"   // wrap_pi

namespace ml4ca {

// Per-launch constants, folded on the host from ml4ca_refmodel_cfg.
struct RefConsts {
  int32_t n_sub;
  float h;
  float hw3[3];   // h w^3
  float hcw2[3];  // h (2 zeta + 1) w^2
  float hcw[3];   // h (2 zeta + 1) w
  float v_max[3], a_max[3];
};

// One env step of one env's filter: x[9] in the row order of the state tensor, updated in place.
__device__ __forceinline__ void refmodel_advance(float (&x)[9], const float (&r)[3], const RefConsts& k) {
#pragma unroll 2
  for (int it = 0; it < k.n_sub; ++it) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      float e = r[d] - x[d];
      if (d == 2) e = wrap_pi(e);
      float a = fmaf(k.hw3[d], e, fmaf(-k.hcw2[d], x[3 + d], fmaf(-k.hcw[d], x[6 + d], x[6 + d])));
      a = fminf(fmaxf(a, -k.a_max[d]), k.a_max[d]);
      float v = fmaf(k.h, a, x[3 + d]);
      v = fminf(fmaxf(v, -k.v_max[d]), k.v_max[d]);
      x[6 + d] = a;
      x[3 + d] = v;
      x[d] = fmaf(k.h, v, x[d]);
    }
  }
}

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

// Jury conditions for the linear sub-step map of one DOF (include/ml4ca_b200.h states them).
static bool substep_stable(double zeta, double omega, double h) {
  const double q = h * omega, c = 2.0 * zeta + 1.0;
  const double a2 = q * q * q + c * q * q + c * q - 3.0, a1 = 3.0 - 2.0 * c * q - c * q * q, a0 = c * q - 1.0;
  const double p1 = 1.0 + a2 + a1 + a0, pm1 = -1.0 + a2 - a1 + a0;
  return p1 > 0.0 && pm1 < 0.0 && fabs(a0) < 1.0 && fabs(a0 * a0 - 1.0) > fabs(a0 * a2 - a1);
}

static int refmodel_consts(const ml4ca_refmodel_cfg* c, RefConsts& k) {
  ML4CA_REQUIRE(c != nullptr, "cfg is NULL");
  ML4CA_REQUIRE(isfinite(c->step_dt) && c->step_dt > 0.f, "step_dt must be finite and > 0");
  for (int d = 0; d < 3; ++d) {
    const float v[] = {c->zeta[d], c->omega[d], c->v_max[d], c->a_max[d]};
    for (float x : v) ML4CA_REQUIRE(isfinite(x) && x > 0.f, "zeta, omega, v_max and a_max must be finite and > 0");
  }
  const double dt = c->step_dt;
  const int n_sub = (int)fmax(1.0, nearbyint(dt / ML4CA_SIM_DT));
  const double h = dt / n_sub;
  for (int d = 0; d < 3; ++d)
    ML4CA_REQUIRE(substep_stable(c->zeta[d], c->omega[d], h),
                  "(zeta, omega, h) make the linear sub-step map unstable (Jury conditions, ml4ca_b200.h)");
  k.n_sub = n_sub;
  k.h = (float)h;
  for (int d = 0; d < 3; ++d) {
    const double w = c->omega[d], cz = 2.0 * (double)c->zeta[d] + 1.0;
    k.hw3[d] = (float)(h * w * w * w);
    k.hcw2[d] = (float)(h * cz * w * w);
    k.hcw[d] = (float)(h * cz * w);
    k.v_max[d] = c->v_max[d];
    k.a_max[d] = c->a_max[d];
  }
  return ML4CA_OK;
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
