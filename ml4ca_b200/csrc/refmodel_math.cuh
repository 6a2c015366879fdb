// refmodel_math.cuh -- the DP reference model's per-env recurrence (refmodel.cu states the model) and its host-side
// configuration, shared by the stand-alone reference-model kernels (refmodel.cu) and the env-step variant that runs the
// model in the loop (env_kernels.cuh, REF = true).
#pragma once
#include <math.h>

#include "common.h"
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

// Jury conditions for the linear sub-step map of one DOF (include/ml4ca_b200.h states them).
static inline bool substep_stable(double zeta, double omega, double h) {
  const double q = h * omega, c = 2.0 * zeta + 1.0;
  const double a2 = q * q * q + c * q * q + c * q - 3.0, a1 = 3.0 - 2.0 * c * q - c * q * q, a0 = c * q - 1.0;
  const double p1 = 1.0 + a2 + a1 + a0, pm1 = -1.0 + a2 - a1 + a0;
  return p1 > 0.0 && pm1 < 0.0 && fabs(a0) < 1.0 && fabs(a0 * a0 - 1.0) > fabs(a0 * a2 - a1);
}

static inline int refmodel_consts(const ml4ca_refmodel_cfg* c, RefConsts& k) {
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
