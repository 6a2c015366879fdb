// pinv_pid.cu -- K2: DP PID controller + fixed-matrix pseudoinverse thrust allocation, one thread per environment.
//
// THE REFERENCE DOES NOT CONTAIN THIS COMPONENT: it lives in DNV GL's private dp_controller ROS package and is
// only referenced (qp_allocator.py:6 "dp_controller/nodesThruster_allocation.py", :83 the tau_controller topic it
// feeds, SupervisedTau.py:37 "Saturation according to dp_controller/DP_PID.py").  The equations below are this
// build's own statement (PARITY UNPINNED, see DESIGN.md); oracle/pinv_oracle.py restates them in float64.
//
//   PID   e = R(psi)^T (eta - ref)[0:2],  e_psi = wrap_rad(psi - psi_ref)
//         I <- clamp(I + dt e, +-sat/Ki)                (anti-windup)
//         tau = clamp(-(Kp e + Kd nu + Ki I), +-[69, 30, 80])
//         with velocity feed-forward (ml4ca_pinv_pid_ff): Kd (nu - R(psi)^T v_d), v_d the reference model's NED rates
//   PINV  extended thrust f = [F1x, F1y, F2x, F2y, F3y] (port, star stern pods; bow fixed at 90 deg),
//         tau = T f with the 3x5 configuration matrix of the reference geometry (qp_allocator.py:69-70),
//         f = T^+ tau (T^+ = T^T (T T^T)^-1, a constant 5x3 matrix), F_i = hypot, alpha_i = atan2,
//         n_i = sign(F_i / K_i) sqrt(|F_i / K_i|) clipped to +-100 % (thrust law qp_allocator.py:284-288).
//
// HBM-bound: 80 algorithmic bytes per env (read eta, nu, ref, I = 48; write I, n, alpha = 32); 92 with feed-forward.
#include <math.h>

#include "common.h"
#include "env_math.cuh"

namespace ml4ca {

struct PinvMatrix {
  float m[5][3];
};

// T^+ in double on the host (3x3 symmetric inverse by cofactors).
static PinvMatrix make_pinv() {
  const double lx1 = ML4CA_LX_PORT, ly1 = ML4CA_LY_PORT, lx2 = ML4CA_LX_STAR, ly2 = ML4CA_LY_STAR, lx3 = ML4CA_LX_BOW;
  const double T[3][5] = {{1, 0, 1, 0, 0}, {0, 1, 0, 1, 1}, {-ly1, lx1, -ly2, lx2, lx3}};
  double G[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      G[i][j] = 0;
      for (int k = 0; k < 5; ++k) G[i][j] += T[i][k] * T[j][k];
    }
  const double det = G[0][0] * (G[1][1] * G[2][2] - G[1][2] * G[2][1]) - G[0][1] * (G[1][0] * G[2][2] - G[1][2] * G[2][0]) +
                     G[0][2] * (G[1][0] * G[2][1] - G[1][1] * G[2][0]);
  double Gi[3][3];
  Gi[0][0] = (G[1][1] * G[2][2] - G[1][2] * G[2][1]) / det;
  Gi[0][1] = (G[0][2] * G[2][1] - G[0][1] * G[2][2]) / det;
  Gi[0][2] = (G[0][1] * G[1][2] - G[0][2] * G[1][1]) / det;
  Gi[1][0] = (G[1][2] * G[2][0] - G[1][0] * G[2][2]) / det;
  Gi[1][1] = (G[0][0] * G[2][2] - G[0][2] * G[2][0]) / det;
  Gi[1][2] = (G[0][2] * G[1][0] - G[0][0] * G[1][2]) / det;
  Gi[2][0] = (G[1][0] * G[2][1] - G[1][1] * G[2][0]) / det;
  Gi[2][1] = (G[0][1] * G[2][0] - G[0][0] * G[2][1]) / det;
  Gi[2][2] = (G[0][0] * G[1][1] - G[0][1] * G[1][0]) / det;
  PinvMatrix P;
  for (int k = 0; k < 5; ++k)
    for (int j = 0; j < 3; ++j) {
      double s = 0;
      for (int i = 0; i < 3; ++i) s += T[i][k] * Gi[i][j];
      P.m[k][j] = (float)s;
    }
  return P;
}

__device__ __forceinline__ float thrust_percent(float F, float K) {
  const float fk = F / K;
  const float n = copysignf(sqrtf(fabsf(fk)), fk);
  return fminf(fmaxf(n, -(float)ML4CA_THRUST_BOUND), (float)ML4CA_THRUST_BOUND);
}

__device__ __forceinline__ void pinv_allocate(const PinvMatrix& P, float tx, float ty, float tn, float& n_port,
                                              float& n_star, float& n_bow, float& a_port, float& a_star) {
  float f[5];
#pragma unroll
  for (int k = 0; k < 5; ++k) f[k] = P.m[k][0] * tx + P.m[k][1] * ty + P.m[k][2] * tn;
  const float F1 = sqrtf(f[0] * f[0] + f[1] * f[1]);
  const float F2 = sqrtf(f[2] * f[2] + f[3] * f[3]);
  a_port = atan2f(f[1], f[0]);
  a_star = atan2f(f[3], f[2]);
  n_port = thrust_percent(F1, (float)ML4CA_K_STERN);
  n_star = thrust_percent(F2, (float)ML4CA_K_STERN);
  n_bow = thrust_percent(f[4], (float)ML4CA_K_BOW);
}

// One env of the PID + allocation step; integ[k] in: I, out: the updated I.  FF: the D-term acts on vel - R(psi)^T vd.
template <bool FF>
__device__ __forceinline__ void pid_one(const PinvMatrix& P, const float (&eta)[3], const float (&vel)[3], const float (&ref)[3],
                                        const float (&vd)[3], float (&integ)[3], float (&tau)[3], float (&npct)[3],
                                        float (&alpha)[2]) {
  const float eN = eta[0] - ref[0], eE = eta[1] - ref[1];
  const float ep = wrap_rad(eta[2] - ref[2]);
  float s, c;
  sincosf(eta[2], &s, &c);
  const float e[3] = {c * eN + s * eE, c * eE - s * eN, ep};
  float dv[3] = {vel[0], vel[1], vel[2]};
  if constexpr (FF) {
    dv[0] = vel[0] - (c * vd[0] + s * vd[1]);
    dv[1] = vel[1] - (c * vd[1] - s * vd[0]);
    dv[2] = vel[2] - vd[2];
  }
  const float kp[3] = {(float)ML4CA_PID_KP_X, (float)ML4CA_PID_KP_Y, (float)ML4CA_PID_KP_N};
  const float kd[3] = {(float)ML4CA_PID_KD_X, (float)ML4CA_PID_KD_Y, (float)ML4CA_PID_KD_N};
  const float ki[3] = {(float)ML4CA_PID_KI_X, (float)ML4CA_PID_KI_Y, (float)ML4CA_PID_KI_N};
  const float sat[3] = {(float)ML4CA_PID_SAT_X, (float)ML4CA_PID_SAT_Y, (float)ML4CA_PID_SAT_N};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float lim = sat[k] / ki[k];
    float I = integ[k] + (float)ML4CA_PID_DT * e[k];
    I = fminf(fmaxf(I, -lim), lim);
    integ[k] = I;
    const float t = -(kp[k] * e[k] + kd[k] * dv[k] + ki[k] * I);
    tau[k] = fminf(fmaxf(t, -sat[k]), sat[k]);
  }
  pinv_allocate(P, tau[0], tau[1], tau[2], npct[0], npct[1], npct[2], alpha[0], alpha[1]);
}

// VEC consecutive envs per thread: with VEC = 2 every row access is 64 bits wide (a warp covers 256 contiguous bytes per
// row), half the load / store instructions per env of the scalar variant (odd n or unaligned rows).  FF reads v_d [3, n],
// the trailing argument (unused without FF, so the FF = false kernels keep the parameter layout of the plain PID).
template <int VEC, bool FF>
__global__ void __launch_bounds__(256) pinv_pid_kernel(int64_t n, const PinvMatrix P, const float* __restrict__ eta,
                                                       const float* __restrict__ nu, const float* __restrict__ ref,
                                                       float* __restrict__ integ, float* __restrict__ tau_out,
                                                       float* __restrict__ n_pct, float* __restrict__ alpha,
                                                       const float* __restrict__ v_d) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  if (i >= n) return;
  float e_[3][VEC], v_[3][VEC], r_[3][VEC], I_[3][VEC], d_[3][VEC];
  auto ld = [&](const float* row, float (&x)[VEC]) {
    if constexpr (VEC == 2) {
      const float2 t = *reinterpret_cast<const float2*>(row + i);
      x[0] = t.x, x[1] = t.y;
    } else {
      x[0] = row[i];
    }
  };
  auto st = [&](float* row, const float (&x)[VEC]) {
    if constexpr (VEC == 2) {
      *reinterpret_cast<float2*>(row + i) = make_float2(x[0], x[1]);
    } else {
      row[i] = x[0];
    }
  };
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    ld(eta + (int64_t)k * n, e_[k]);
    ld(nu + (int64_t)k * n, v_[k]);
    ld(ref + (int64_t)k * n, r_[k]);
    ld(integ + (int64_t)k * n, I_[k]);
    if constexpr (FF) ld(v_d + (int64_t)k * n, d_[k]);
  }
  float tau[3][VEC], np_[3][VEC], al_[2][VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    const float e1[3] = {e_[0][j], e_[1][j], e_[2][j]}, v1[3] = {v_[0][j], v_[1][j], v_[2][j]}, r1[3] = {r_[0][j], r_[1][j], r_[2][j]};
    float I1[3] = {I_[0][j], I_[1][j], I_[2][j]}, t1[3], n1[3], a1[2], d1[3] = {0.f, 0.f, 0.f};
    if constexpr (FF) d1[0] = d_[0][j], d1[1] = d_[1][j], d1[2] = d_[2][j];
    pid_one<FF>(P, e1, v1, r1, d1, I1, t1, n1, a1);
#pragma unroll
    for (int k = 0; k < 3; ++k) I_[k][j] = I1[k], tau[k][j] = t1[k], np_[k][j] = n1[k];
    al_[0][j] = a1[0], al_[1][j] = a1[1];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    st(integ + (int64_t)k * n, I_[k]);
    if (tau_out != nullptr) st(tau_out + (int64_t)k * n, tau[k]);
    st(n_pct + (int64_t)k * n, np_[k]);
  }
  st(alpha, al_[0]);
  st(alpha + n, al_[1]);
}

__global__ void __launch_bounds__(256) pinv_allocate_kernel(int64_t n, const PinvMatrix P,
                                                            const float* __restrict__ tau,
                                                            float* __restrict__ n_pct, float* __restrict__ alpha) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float np_, ns_, nb_, ap_, as_;
  pinv_allocate(P, tau[i], tau[n + i], tau[2 * n + i], np_, ns_, nb_, ap_, as_);
  n_pct[i] = np_, n_pct[n + i] = ns_, n_pct[2 * n + i] = nb_;
  alpha[i] = ap_, alpha[n + i] = as_;
}

}  // namespace ml4ca

using namespace ml4ca;

extern "C" {

}  // extern "C"

namespace {

template <bool FF>
int launch_pinv_pid(int64_t n, const float* eta, const float* nu, const float* ref, const float* v_d, float* integ,
                    float* tau, float* n_pct, float* alpha, void* stream) {
  if (n == 0) return ML4CA_OK;
  static const PinvMatrix P = make_pinv();
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto al8 = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 7u) == 0; };
  if (n % 2 == 0 && al8(eta) && al8(nu) && al8(ref) && al8(integ) && al8(tau) && al8(n_pct) && al8(alpha) && al8(v_d)) {
    pinv_pid_kernel<2, FF><<<(unsigned)((n / 2 + 255) / 256), 256, 0, st>>>(n, P, eta, nu, ref, integ, tau, n_pct, alpha, v_d);
  } else {
    pinv_pid_kernel<1, FF><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, P, eta, nu, ref, integ, tau, n_pct, alpha, v_d);
  }
  return check_launch("pinv_pid_kernel");
}

}  // namespace

extern "C" {

int ml4ca_pinv_pid(int64_t n, const float* eta, const float* nu, const float* ref, float* integ, float* tau,
                   float* n_pct, float* alpha, void* stream) {
  ML4CA_REQUIRE(n >= 0 && eta && nu && ref && integ && n_pct && alpha, "bad arguments");
  return launch_pinv_pid<false>(n, eta, nu, ref, nullptr, integ, tau, n_pct, alpha, stream);
}

int ml4ca_pinv_pid_ff(int64_t n, const float* eta, const float* nu, const float* ref, const float* v_d, float* integ,
                      float* tau, float* n_pct, float* alpha, void* stream) {
  ML4CA_REQUIRE(n >= 0 && eta && nu && ref && v_d && integ && n_pct && alpha, "bad arguments");
  return launch_pinv_pid<true>(n, eta, nu, ref, v_d, integ, tau, n_pct, alpha, stream);
}

int ml4ca_pinv_allocate(int64_t n, const float* tau, float* n_pct, float* alpha, void* stream) {
  ML4CA_REQUIRE(n >= 0 && tau && n_pct && alpha, "bad arguments");
  if (n == 0) return ML4CA_OK;
  static const PinvMatrix P = make_pinv();
  pinv_allocate_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, P, tau, n_pct,
                                                                                                  alpha);
  return check_launch("pinv_allocate_kernel");
}

}  // extern "C"
