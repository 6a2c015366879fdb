// env_kernels.cuh -- K3: batched Revolt.reset / Revolt.step for millions of independent environments.
//
// Replaces /root/reference/src/rl/windows_workspace/specific/customEnv.py:92-133 (step) and :135-194 (reset):
// action transform -> thruster commands -> 20 sub-steps of the stand-in 3-DOF hull (in place of the six py4j
// round trips into the Cybersea JVM, customEnv.py:117-124) -> body-frame error -> observation, reward,
// termination, episode-length cut, optional in-kernel re-sampling of finished envs.
//
// Data layout in HBM: struct-of-arrays fp32, one row per state component, row length n_env:
//   eta[3] nu[3] ref[3] prev_thrust[3] angles[3]  +  int32 ep_len, episode
// One thread owns VEC consecutive environments.  The shipped default is VEC = 2: every row access is one 64-bit, fully
// coalesced LDG/STG (a warp touches 256 contiguous bytes per row) and the pair of envs runs the hull sub-steps on the
// packed FP32 pipe (FFMA2, integrate_hull2); VEC = 4 (128-bit rows) and VEC = 1 (unaligned batches) are also
// instantiated (env_step_inst.cu picks).  There is no reuse between environments, so nothing is
// staged through shared memory here; the kernel streams 177 algorithmic bytes per env-step (RevoltFinal,
// extended state, continuous angles: read 60 state + 28 action, write 48 state + 36 obs + 4 rew + 1 done).
// Grid: enough 256-thread CTAs to cover n_env, rounded so that the last wave is full where possible.
#pragma once
#include <new>

#include "common.h"
#include "env_math.cuh"
#include "observer_math.cuh"
#include "refmodel_math.cuh"

#ifndef ML4CA_ENV_MIN_BLOCKS
#define ML4CA_ENV_MIN_BLOCKS 6  // scalar-row kernel: 40 registers, 48 resident warps/SM (measured best on B200)
#endif

#ifndef ML4CA_ENV_MIN_BLOCKS2
#define ML4CA_ENV_MIN_BLOCKS2 3  // two-env packed kernel: 78 registers without spills (4 CTAs = 64 registers spill 72 B:
                                 // 0.514 ms against 0.504 ms per 16 Mi envs over 200 steps)
#endif

#ifndef ML4CA_ENV_MIN_BLOCKS_DIST
#define ML4CA_ENV_MIN_BLOCKS_DIST 4  // disturbed step: 64 registers; 40 would spill around the Philox / Box-Muller draws
#endif

#ifndef ML4CA_ENV_MIN_BLOCKS_WAVE
#define ML4CA_ENV_MIN_BLOCKS_WAVE 4  // step with wave motion: 64 registers, no spills
#endif

#ifndef ML4CA_ENV_MIN_BLOCKS_WAVE_DIST
#define ML4CA_ENV_MIN_BLOCKS_WAVE_DIST 3  // wave motion and disturbance together: 4 CTAs (64 registers) would spill 12-16 B
#endif

#ifndef ML4CA_ENV_MIN_BLOCKS_OBSV
#define ML4CA_ENV_MIN_BLOCKS_OBSV 2  // step with the observer in the loop (any LAG / DIST / WAVE / REF): at most 128 registers
#endif                              // (94-118 with the reference model as well, no spills)

#ifndef ML4CA_ENV_MIN_BLOCKS_REF
#define ML4CA_ENV_MIN_BLOCKS_REF 3  // step with the reference model in the loop, no observer (any LAG / DIST / WAVE): 63-79
                                    // registers, no spills; 4 CTAs (64 registers) spill 4-28 B in the WAVE variants
#endif

namespace ml4ca {

struct EnvParams {
  float* eta;          // [3, n]
  float* nu;           // [3, n]
  float* ref;          // [3, n]
  float* prev_thrust;  // [3, n]
  float* angles;       // [3, n] bow, port, star
  float* obs_tail;     // [3, n] tail (prev_thrust / 100) of the observation a reset returned (ml4ca_env_observe)
  float* cut_obs;      // [obs_dim, n] caller-owned, nullable (ml4ca_env_set_cut_obs): the observation an env returned at its
                       // episode-length cut, saved before the in-kernel restart replaces it (ppo.py:311 evaluates V on it)
  float* tau_act;      // [3, n] lagged thruster wrench (N, N, Nm); read and written only when cfg.actuator_lag_s > 0
  int32_t* ep_len;     // [n] episode word: episode counter << 16 | steps in this episode (env_math.cuh)
  int64_t n;
  float bounds[6];
  float reset_scale[6];
  float inv_step_dt, pad1;
  HullConsts hull;
  int32_t n_sub, max_ep_len;
  int32_t auto_reset, reset_acts;  // reset_acts: customEnv.py:179-188
  uint64_t seed;
  int64_t env_off;
  // one launch may cover a slice [first, first + count) of the batch (host-buffer pipeline, env_step.cu): the state
  // pointers above are then advanced by `first` (row stride stays n) and the caller's action / obs rows have
  // their own stride io_stride.  Whole-batch launches: count = io_stride = n.
  int64_t count, io_stride;
};

// Wave-frequency motion (ml4ca_env_set_waves): the step kernel's last argument, after DistParams, for the reason given
// there (and appended to DistParams it would grow the stack copy the DIST kernels make of it).  The three pointers are
// NULL while waves are off.
struct WaveParams {
  float* motion;       // [3, n] x: surge (m), sway (m), yaw (rad), body frame
  float* rate;         // [3, n] x' (m/s, m/s, rad/s)
  float* omega;        // [n] peak frequency w0 of the episode (rad/s)
  WaveConsts k;
};

// Environmental disturbance (ml4ca_env_set_disturbance).  Passed as the LAST argument of the step kernel rather than
// inside EnvParams: the arguments of the kernels without disturbance then keep their parameter-bank offsets, and
// their code stays what it was.  Both pointers are NULL while no disturbance is enabled.
struct DistParams {
  float* current;      // [2, n] NED current (m/s) of the episode
  float* bias;         // [3, n] NED bias force (N, N, Nm)
  DistConsts k;
};

// DP observer in the loop (ml4ca_env_set_observer): the step kernel's last argument, after WaveParams, for the reason given
// at DistParams.  Both pointers belong to the caller; state is NULL while no observer is attached.
struct ObserverParams {
  float* state;        // [15, n] rows xi1^, xi2^, eta^, nu^, b^ (observer_math.cuh)
  const float* omega;  // [n] w_o (rad/s), clamped by the kernel
  ObsConsts k;
};

// DP reference model in the loop (ml4ca_env_set_refmodel): the step kernel's last argument, after ObserverParams, for the
// reason given at DistParams.  state belongs to the caller and is NULL while no model is attached.
struct RefParams {
  float* state;        // [9, n] rows eta_d, v_d, a_d (refmodel_math.cuh)
  RefConsts k;
};

}  // namespace ml4ca

namespace ml4ca {
// Device staging and streams of ml4ca_env_step_host (created on first use).
struct HostPipe {
  int64_t chunk = 0;           // envs per pipeline stage
  void* slab = nullptr;
  float* act[2];
  float* obs[2];
  float* rew[2];
  uint8_t* done[2];
  cudaStream_t s_in, s_k, s_out;
  cudaEvent_t ev_start, ev_in[2], ev_k[2], ev_out[2];
};
}  // namespace ml4ca

struct ml4ca_env {
  ml4ca_env_cfg cfg;
  int64_t n;
  int32_t device;
  void* slab;
  ml4ca::HostPipe* pipe = nullptr;
  void* dist_slab = nullptr;  // current [2, n] + bias [3, n] rows, allocated when a disturbance is first enabled
  void* wave_slab = nullptr;  // motion [3, n] + rate [3, n] + omega [n] rows, allocated when waves are first enabled
  bool tail_valid;     // obs_tail rows describe the last returned observation (true after a reset, false after a step)
  ml4ca::EnvParams p;
  ml4ca::DistParams dist = {};
  ml4ca::WaveParams wave = {};
  ml4ca::ObserverParams obsv = {};
  ml4ca::RefParams refm = {};
};

namespace ml4ca {

// ---- vector row access -----------------------------------------------------------------------------------------
template <int VEC>
__device__ __forceinline__ void ld_row(const float* __restrict__ row, int64_t i, float (&x)[VEC]) {
  if constexpr (VEC == 4) {
    const float4 t = *reinterpret_cast<const float4*>(row + i);
    x[0] = t.x, x[1] = t.y, x[2] = t.z, x[3] = t.w;
  } else if constexpr (VEC == 2) {
    const float2 t = *reinterpret_cast<const float2*>(row + i);
    x[0] = t.x, x[1] = t.y;
  } else {
    x[0] = row[i];
  }
}
template <int VEC>
__device__ __forceinline__ void ld_row_nc(const float* __restrict__ row, int64_t i, float (&x)[VEC]) {
  if constexpr (VEC == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(row + i));
    x[0] = t.x, x[1] = t.y, x[2] = t.z, x[3] = t.w;
  } else if constexpr (VEC == 2) {
    const float2 t = __ldg(reinterpret_cast<const float2*>(row + i));
    x[0] = t.x, x[1] = t.y;
  } else {
    x[0] = __ldg(row + i);
  }
}
template <int VEC>
__device__ __forceinline__ void st_row(float* __restrict__ row, int64_t i, const float (&x)[VEC]) {
  if constexpr (VEC == 4) {
    *reinterpret_cast<float4*>(row + i) = make_float4(x[0], x[1], x[2], x[3]);
  } else if constexpr (VEC == 2) {
    *reinterpret_cast<float2*>(row + i) = make_float2(x[0], x[1]);
  } else {
    row[i] = x[0];
  }
}
template <int VEC>
__device__ __forceinline__ void ld_irow(const int32_t* __restrict__ row, int64_t i, int32_t (&x)[VEC]) {
  if constexpr (VEC == 4) {
    const int4 t = *reinterpret_cast<const int4*>(row + i);
    x[0] = t.x, x[1] = t.y, x[2] = t.z, x[3] = t.w;
  } else if constexpr (VEC == 2) {
    const int2 t = *reinterpret_cast<const int2*>(row + i);
    x[0] = t.x, x[1] = t.y;
  } else {
    x[0] = row[i];
  }
}
template <int VEC>
__device__ __forceinline__ void st_irow(int32_t* __restrict__ row, int64_t i, const int32_t (&x)[VEC]) {
  if constexpr (VEC == 4) {
    *reinterpret_cast<int4*>(row + i) = make_int4(x[0], x[1], x[2], x[3]);
  } else if constexpr (VEC == 2) {
    *reinterpret_cast<int2*>(row + i) = make_int2(x[0], x[1]);
  } else {
    row[i] = x[0];
  }
}
template <int VEC>
__device__ __forceinline__ void st_flags(uint8_t* __restrict__ row, int64_t i, const uint32_t (&x)[VEC]) {
  if constexpr (VEC == 4) {
    *reinterpret_cast<uint32_t*>(row + i) = x[0] | (x[1] << 8) | (x[2] << 16) | (x[3] << 24);
  } else if constexpr (VEC == 2) {
    *reinterpret_cast<uint16_t*>(row + i) = (uint16_t)(x[0] | (x[1] << 8));
  } else {
    row[i] = (uint8_t)x[0];
  }
}

// ---- K3 ------------------------------------------------------------------------------------------------------------
// LAG = true (one env per thread only): the wrench lag of cfg.actuator_lag_s, three more state rows in and out.
// DIST = true (one env per thread only): the ocean current and the bias force of ml4ca_env_set_disturbance.  The hull
// recurrence runs unchanged on the velocity relative to the water, nu_r = nu - R(psi0)^T v_c, with the bias added to
// the wrench as R(psi0)^T b (after the lag); the pose then drifts by n_sub h v_c and nu = nu_r + R(psi1)^T v_c is the
// velocity over ground again.  20 B more read (current, bias) and 12 B more written (bias) per env-step: 209 B.
// WAVE = true (one env per thread only): the wave-frequency motion of ml4ca_env_set_waves.  After the hull step the wave
// state takes one exact step (advance_waves), and the observation, reward and termination are computed from the measured
// pose and velocity (add_wave_motion) instead of the LF state, which is stored unchanged.  28 B more read (x, x', w0)
// and 24 B more written (x, x') per env-step: 229 B, 261 B together with the disturbance.
// OBSV = true (one env per thread only): the DP observer of ml4ca_env_set_observer runs in the loop.  Its column takes one
// step (observer_advance) on the measured pose after this step and the thrust and azimuths this step applied, and
// observation rows 0-5 become error_frame(eta^, ref) and nu^; rows 6-8, the reward, the flags and the env state are
// those of the kernel without it.  cut_obs is the estimate-based observation before the restart; a restart re-initialises
// the column from the new episode's measured pose (nu^ = 0 in the returned observation).  124 B more per env-step
// (read 60 + 4, write 60): 301 B for RevoltFinal (extended, continuous angles), 353 B in waves.
// REF = true (one env per thread only): the DP reference model of ml4ca_env_set_refmodel runs in the loop.  Its column
// first takes one step (refmodel_advance) on the set-point rows s, and everything the step forms against the set-point
// then uses eta_d(t+1) instead: observation rows 0-2 (and the observer's error frame), the reward and the termination.
// cut_obs is formed after the advance and before the restart; a restart starts the column again at the new episode's LF
// pose (eta_d = eta, v_d = a_d = 0).  72 B more per env-step (read 36, write 36; s is read anyway): 249 B for RevoltFinal
// (extended, continuous angles), 373 B with the observer.
template <int KIND, bool CONT, bool EXT, int VEC, bool LAG = false, bool DIST = false, bool WAVE = false, bool OBSV = false,
          bool REF = false>
__global__ void __launch_bounds__(256, OBSV ? ML4CA_ENV_MIN_BLOCKS_OBSV : (REF ? ML4CA_ENV_MIN_BLOCKS_REF : (WAVE ? (DIST ? ML4CA_ENV_MIN_BLOCKS_WAVE_DIST : ML4CA_ENV_MIN_BLOCKS_WAVE) : (DIST ? ML4CA_ENV_MIN_BLOCKS_DIST : (VEC == 1 ? ML4CA_ENV_MIN_BLOCKS : (VEC == 2 ? ML4CA_ENV_MIN_BLOCKS2 : 1)))))) env_step_kernel(const EnvParams p, const float* __restrict__ action,
                                                       float* __restrict__ obs, float* __restrict__ rew,
                                                       uint8_t* __restrict__ done, const DistParams d,
                                                       const WaveParams wv, const ObserverParams ob,
                                                       const RefParams rf) {
  using T = EnvTraits<KIND, CONT>;
  static_assert(!LAG || VEC == 1, "the lagged integrator is scalar");
  static_assert(!DIST || VEC == 1, "the disturbed step is scalar");
  static_assert(!WAVE || VEC == 1, "the step with wave motion is scalar");
  static_assert(!OBSV || VEC == 1, "the step with the observer in the loop is scalar");
  static_assert(!REF || VEC == 1, "the step with the reference model in the loop is scalar");
  const int64_t n = p.n, ios = p.io_stride;
  const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  if (i0 >= p.count) return;

  // ---- loads: issue everything up front so that ~20 independent 128-bit requests are in flight per thread ----
  float a[T::ACT][VEC];
#pragma unroll
  for (int c = 0; c < T::ACT; ++c) ld_row_nc<VEC>(action + (int64_t)c * ios, i0, a[c]);
  float eta[3][VEC], nu[3][VEC], ref[3][VEC], pth[3][VEC], ang[3][VEC];
  int32_t ep[VEC];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    ld_row<VEC>(p.eta + (int64_t)c * n, i0, eta[c]);
    ld_row<VEC>(p.nu + (int64_t)c * n, i0, nu[c]);
    ld_row<VEC>(p.ref + (int64_t)c * n, i0, ref[c]);
    if constexpr (EXT) ld_row<VEC>(p.prev_thrust + (int64_t)c * n, i0, pth[c]);
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const bool is_state = (T::NANG == 3) || (T::NANG == 2 && c > 0);
    if (is_state) {
      ld_row<VEC>(p.angles + (int64_t)c * n, i0, ang[c]);
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) ang[c][j] = (c == 0) ? T::DEF_BOW : (c == 1 ? T::DEF_PORT : T::DEF_STAR);
    }
  }
  ld_irow<VEC>(p.ep_len, i0, ep);
  float tact[3][VEC];
  if constexpr (LAG) {
#pragma unroll
    for (int c = 0; c < 3; ++c) ld_row<VEC>(p.tau_act + (int64_t)c * n, i0, tact[c]);
  }
  float cur[2][VEC], bia[3][VEC];
  if constexpr (DIST) {
#pragma unroll
    for (int c = 0; c < 2; ++c) ld_row<VEC>(d.current + (int64_t)c * n, i0, cur[c]);
#pragma unroll
    for (int c = 0; c < 3; ++c) ld_row<VEC>(d.bias + (int64_t)c * n, i0, bia[c]);
  }
  float wm[3], wr[3], w0 = 0.f;                                        // VEC == 1 when WAVE
  if constexpr (WAVE) {
#pragma unroll
    for (int c = 0; c < 3; ++c) wm[c] = wv.motion[(int64_t)c * n + i0], wr[c] = wv.rate[(int64_t)c * n + i0];
    w0 = wv.omega[i0];
  }
  float ox[15], wo = 0.f;                                              // VEC == 1 when OBSV
  if constexpr (OBSV) {
#pragma unroll
    for (int r = 0; r < 15; ++r) ox[r] = ob.state[(int64_t)r * n + i0];
    wo = clamp_omega(ob.omega[i0]);
  }
  float rx[9];                                                         // VEC == 1 when REF
  if constexpr (REF) {
#pragma unroll
    for (int q = 0; q < 9; ++q) rx[q] = rf.state[(int64_t)q * n + i0];
  }

  float o[9][VEC], rw[VEC];
  uint32_t flags[VEC];
  bool any_reset = false;
  // ---- phase A: action transform, azimuth commands, thruster wrench ------------------------------------------------
  float thr[3][VEC], dang[3][VEC], wx[VEC], wy[VEC], wn[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    float act[T::ACT], cmd[T::NCMD];
    int sat[T::NCMD];
#pragma unroll
    for (int c = 0; c < T::ACT; ++c) act[c] = a[c][j];
    float sp = 0.f, cp = 1.f, ss = 0.f, cs = 1.f;
    if constexpr (KIND == ML4CA_ENV_FINAL && CONT) {
      transform_action_final_cont(act, cmd, sat, sp, cp, ss, cs);      // customEnv.py:104-110, (sin, cos) from the pairs
    } else {
      transform_action<KIND, CONT>(act, cmd, sat);
    }
    const float pa_bow = ang[0][j], pa_port = ang[1][j], pa_star = ang[2][j];  // prev_angles, :102
    apply_angle_commands<KIND, CONT>(cmd, ang[0][j], ang[1][j], ang[2][j]);    // :117-122
    dang[0][j] = ang[0][j] - pa_bow, dang[1][j] = ang[1][j] - pa_port, dang[2][j] = ang[2][j] - pa_star;
    thr[0][j] = cmd[0], thr[1][j] = cmd[1], thr[2][j] = cmd[2];        // prev_thrust <- action[0:3], :126
    wx[j] = wy[j] = wn[j] = 0.f;
    if (p.n_sub > 0) {
      float sb, cb;
      if constexpr (T::NANG == 3) {
        sincosf(ang[0][j], &sb, &cb);
      } else if constexpr (KIND == ML4CA_ENV_SIMPLE) {
        sincosf(T::DEF_BOW, &sb, &cb);
      } else {
        sb = 1.f, cb = 0.f;                                            // bow azimuth fixed at 90 deg (:394-399)
      }
      if constexpr (!(KIND == ML4CA_ENV_FINAL && CONT)) {
        sincosf(ang[1][j], &sp, &cp);
        sincosf(ang[2][j], &ss, &cs);
      }
      thruster_wrench_sc(cmd[0], cmd[1], cmd[2], sb, cb, sp, cp, ss, cs, wx[j], wy[j], wn[j]);
    }
  }
  // ---- phase B: dTwin.step(n_steps), :124 ---------------------------------------------------------------------------
  if (p.n_sub > 0) {
    if constexpr (DIST) {                                              // VEC == 1
      const float cN = cur[0][0], cE = cur[1][0];
      float s0, c0;
      sincos_heading(eta[2][0], s0, c0);
      nu[0][0] -= fmaf(c0, cN, s0 * cE);                               // nu_r = nu - R(psi0)^T v_c
      nu[1][0] -= fmaf(c0, cE, -s0 * cN);
      const float fx = fmaf(c0, bia[0][0], s0 * bia[1][0]);            // R(psi0)^T b, held over the sub-steps
      const float fy = fmaf(c0, bia[1][0], -s0 * bia[0][0]);
      if constexpr (LAG) {
        integrate_hull_lag<true>(eta[0][0], eta[1][0], eta[2][0], nu[0][0], nu[1][0], nu[2][0], wx[0], wy[0], wn[0],
                                 tact[0][0], tact[1][0], tact[2][0], p.n_sub, p.hull, fx, fy, bia[2][0]);
      } else {
        integrate_hull(eta[0][0], eta[1][0], eta[2][0], nu[0][0], nu[1][0], nu[2][0], wx[0] + fx, wy[0] + fy,
                       wn[0] + bia[2][0], p.n_sub, p.hull);
      }
      eta[0][0] = fmaf(d.k.t_step, cN, eta[0][0]);                  // + n_sub h v_c
      eta[1][0] = fmaf(d.k.t_step, cE, eta[1][0]);
      float s1, c1;
      sincos_heading(eta[2][0], s1, c1);
      nu[0][0] += fmaf(c1, cN, s1 * cE);                               // back to the velocity over ground
      nu[1][0] += fmaf(c1, cE, -s1 * cN);
    } else if constexpr (LAG) {
      integrate_hull_lag(eta[0][0], eta[1][0], eta[2][0], nu[0][0], nu[1][0], nu[2][0], wx[0], wy[0], wn[0], tact[0][0],
                         tact[1][0], tact[2][0], p.n_sub, p.hull);
    } else if constexpr (VEC == 2) {                                   // two envs per thread: packed FP32 pipe
      float2 N = make_float2(eta[0][0], eta[0][1]), E = make_float2(eta[1][0], eta[1][1]),
             psi = make_float2(eta[2][0], eta[2][1]), u = make_float2(nu[0][0], nu[0][1]),
             v = make_float2(nu[1][0], nu[1][1]), r = make_float2(nu[2][0], nu[2][1]);
      integrate_hull2(N, E, psi, u, v, r, make_float2(wx[0], wx[1]), make_float2(wy[0], wy[1]),
                      make_float2(wn[0], wn[1]), p.n_sub, p.hull);
      eta[0][0] = N.x, eta[0][1] = N.y, eta[1][0] = E.x, eta[1][1] = E.y, eta[2][0] = psi.x, eta[2][1] = psi.y;
      nu[0][0] = u.x, nu[0][1] = u.y, nu[1][0] = v.x, nu[1][1] = v.y, nu[2][0] = r.x, nu[2][1] = r.y;
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j)
        integrate_hull(eta[0][j], eta[1][j], eta[2][j], nu[0][j], nu[1][j], nu[2][j], wx[j], wy[j], wn[j], p.n_sub,
                       p.hull);
    }
  }
  // ---- phase C: observation, reward, termination --------------------------------------------------------------------
  if constexpr (WAVE) advance_waves(p.seed, p.env_off + i0, ep[0] + 1, wv.k, w0, wm, wr);   // word after this step
  if constexpr (REF) {                 // eta_d(t) -> eta_d(t+1) on s; from here on the step forms everything against eta_d
    const float s[3] = {ref[0][0], ref[1][0], ref[2][0]};
    refmodel_advance(rx, s, rf.k);
    ref[0][0] = rx[0], ref[1][0] = rx[1], ref[2][0] = rx[2];
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    float mN = eta[0][j], mE = eta[1][j], mP = eta[2][j], mu = nu[0][j], mv = nu[1][j], mr = nu[2][j];
    if constexpr (WAVE) add_wave_motion(mN, mE, mP, mu, mv, mr, wm, wr);       // the measured pose and velocity
    float xb, yb, pb;                                                  // state_extended(), :125
    error_frame(mN, mE, mP, ref[0][j], ref[1][j], ref[2][j], xb, yb, pb);
    o[0][j] = xb, o[1][j] = yb, o[2][j] = pb;
    o[3][j] = mu, o[4][j] = mv, o[5][j] = mr;
    float old_thrust[3] = {0.f, 0.f, 0.f};
    if constexpr (EXT) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        old_thrust[c] = pth[c][j];
        o[6 + c][j] = div100(pth[c][j]);                               // prev_thrust / 100.0, :204 (bit-exact)
      }
    }
    const float thrust[3] = {thr[0][j], thr[1][j], thr[2][j]};
    rw[j] = reward_fn<EXT>(xb, yb, pb, mu, mv, mr, thrust, old_thrust, dang[0][j], dang[1][j], dang[2][j], p.inv_step_dt,
                           1.0f / T::ANG_BOUND);                                                   // :128
    const bool term = is_terminal(xb, yb, pb, mu, mv, mr, p.bounds);                             // :129
    ep[j] += 1;                                                        // low half: steps in this episode
    const bool trunc = (int32_t)((uint32_t)ep[j] & kEpLenMask) >= p.max_ep_len;   // ppo.py:304
    flags[j] = (term ? ML4CA_DONE_TERMINAL : 0u) | (trunc ? ML4CA_DONE_TRUNCATED : 0u);
    if constexpr (OBSV) {         // y = the measured pose; tau from the thrust and azimuths this step applied
      const float y[3] = {mN, mE, mP};
      float sb, cb, sp, cp, ss, cs, tx, ty, tn;
      sincosf(ang[0][j], &sb, &cb);
      sincosf(ang[1][j], &sp, &cp);
      sincosf(ang[2][j], &ss, &cs);
      thruster_wrench_sc(thr[0][j], thr[1][j], thr[2][j], sb, cb, sp, cp, ss, cs, tx, ty, tn);
      observer_advance(ox, y, tx, ty, tn, wo, ob.k);
      error_frame(ox[6], ox[7], ox[8], ref[0][j], ref[1][j], ref[2][j], o[0][j], o[1][j], o[2][j]);
      o[3][j] = ox[9], o[4][j] = ox[10], o[5][j] = ox[11];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) pth[c][j] = thrust[c];
    any_reset |= (flags[j] != 0u);
  }
  if constexpr (DIST) {                                                // the step applied b's value at its start
    if (d.k.gm) advance_bias(p.seed, p.env_off + i0, ep[0], d.k, bia[0][0], bia[1][0], bia[2][0]);
  }

  if (p.auto_reset && any_reset) {  // rare (1 / episode length): keeps the RNG off the common path
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      if (flags[j] == 0u) continue;
      if (flags[j] == ML4CA_DONE_TRUNCATED && p.cut_obs != nullptr) {   // o2 of ppo.py:293 at the cut: the bootstrap input
#pragma unroll
        for (int c = 0; c < (EXT ? 9 : 6); ++c) p.cut_obs[(int64_t)c * n + i0 + j] = o[c][j];
      }
      sample_reset(p.seed, p.env_off + i0 + j, ep[j], p.reset_scale, eta[0][j], eta[1][j], eta[2][j], nu[0][j],
                   nu[1][j], nu[2][j]);
      ang[0][j] = T::DEF_BOW, ang[1][j] = T::DEF_PORT, ang[2][j] = T::DEF_STAR;
      if constexpr (LAG) tact[0][j] = tact[1][j] = tact[2][j] = 0.f;
      if constexpr (DIST) {                                            // a new current and bias (old episode word)
        float cj[2], bj[3];
        sample_disturbance(p.seed, p.env_off + i0 + j, ep[j], d.k, cj, bj);
        d.current[i0 + j] = cj[0], d.current[n + i0 + j] = cj[1];
        bia[0][j] = bj[0], bia[1][j] = bj[1], bia[2][j] = bj[2];
      }
      float mN = eta[0][j], mE = eta[1][j], mP = eta[2][j], mu = nu[0][j], mv = nu[1][j], mr = nu[2][j];
      if constexpr (WAVE) {                                            // a new w0 and a stationary draw (old episode word)
        float xj[3], xdj[3], wj;
        sample_waves(p.seed, p.env_off + i0 + j, ep[j], wv.k.sigma[0], wv.k.sigma[1], wv.k.sigma[2], wv.k.omega_lo,
                     wv.k.omega_span, xj, xdj, &wj);
        wv.omega[i0 + j] = wj;
#pragma unroll
        for (int c = 0; c < 3; ++c) wm[c] = xj[c], wr[c] = xdj[c];
        add_wave_motion(mN, mE, mP, mu, mv, mr, wm, wr);
      }
      if constexpr (REF) {                                             // eta_d = the new LF pose, v_d = a_d = 0
#pragma unroll
        for (int q = 0; q < 9; ++q) rx[q] = q < 3 ? eta[q][j] : 0.f;
        ref[0][j] = rx[0], ref[1][j] = rx[1], ref[2][j] = rx[2];
      }
      float t0[3] = {0.f, 0.f, 0.f};                                   // customEnv.py:190
      if (p.reset_acts) sample_reset_thrust(p.seed, p.env_off + i0 + j, ep[j], t0);   // :179-188 (old episode word)
      ep[j] = next_episode_word(ep[j]);
      pth[0][j] = t0[0], pth[1][j] = t0[1], pth[2][j] = t0[2];
      error_frame(mN, mE, mP, ref[0][j], ref[1][j], ref[2][j], o[0][j], o[1][j], o[2][j]);
      o[3][j] = mu, o[4][j] = mv, o[5][j] = mr;
      if constexpr (EXT) o[6][j] = div100(t0[0]), o[7][j] = div100(t0[1]), o[8][j] = div100(t0[2]);
      if constexpr (OBSV) {                                            // eta^ = y of the new episode, the rest 0
        const float y[3] = {mN, mE, mP};
        observer_reset_column(ox, y);
        o[3][j] = o[4][j] = o[5][j] = 0.f;
      }
    }
  }

  // ---- stores ---------------------------------------------------------------------------------------------------
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    st_row<VEC>(p.eta + (int64_t)c * n, i0, eta[c]);
    st_row<VEC>(p.nu + (int64_t)c * n, i0, nu[c]);
    st_row<VEC>(p.prev_thrust + (int64_t)c * n, i0, pth[c]);
    const bool is_state = (T::NANG == 3) || (T::NANG == 2 && c > 0);
    if (is_state) st_row<VEC>(p.angles + (int64_t)c * n, i0, ang[c]);
  }
  st_irow<VEC>(p.ep_len, i0, ep);
  if constexpr (LAG) {
#pragma unroll
    for (int c = 0; c < 3; ++c) st_row<VEC>(p.tau_act + (int64_t)c * n, i0, tact[c]);
  }
  if constexpr (DIST) {
#pragma unroll
    for (int c = 0; c < 3; ++c) st_row<VEC>(d.bias + (int64_t)c * n, i0, bia[c]);
  }
  if constexpr (WAVE) {
#pragma unroll
    for (int c = 0; c < 3; ++c) wv.motion[(int64_t)c * n + i0] = wm[c], wv.rate[(int64_t)c * n + i0] = wr[c];
  }
  if constexpr (OBSV) {
#pragma unroll
    for (int r = 0; r < 15; ++r) ob.state[(int64_t)r * n + i0] = ox[r];
  }
  if constexpr (REF) {
#pragma unroll
    for (int q = 0; q < 9; ++q) rf.state[(int64_t)q * n + i0] = rx[q];
  }
#pragma unroll
  for (int c = 0; c < (EXT ? 9 : 6); ++c) st_row<VEC>(obs + (int64_t)c * ios, i0, o[c]);
  st_row<VEC>(rew, i0, rw);
  st_flags<VEC>(done, i0, flags);
}

// ---- reset ----------------------------------------------------------------------------------------------------------
// mask nullable; explicit eta/nu (reset_to) or Philox sampling.  Writes obs for the reset envs only.  With an observer
// attached, the reset columns of its state start from the measured pose (eta^ = y, the rest 0) and obs rows 3-5 are nu^ = 0.
// With a reference model attached, the reset columns of its state start from the LF pose (eta_d = eta, v_d = a_d = 0) and
// obs rows 0-2 are formed against that eta_d.
template <int KIND, bool CONT, bool EXT>
__global__ void __launch_bounds__(256) env_reset_kernel(const EnvParams p, const uint8_t* __restrict__ mask,
                                                        const float* __restrict__ eta_in,
                                                        const float* __restrict__ nu_in,
                                                        float* __restrict__ obs, const DistParams d,
                                                        const WaveParams wv, const ObserverParams ob,
                                                        const RefParams rf) {
  using T = EnvTraits<KIND, CONT>;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  if (mask != nullptr && mask[i] == 0) return;
  const int64_t n = p.n;
  float N, E, psi, u, v, r;
  const int32_t epi = p.ep_len[i];
  if (eta_in != nullptr) {
    N = eta_in[i], E = eta_in[n + i], psi = eta_in[2 * n + i];
    u = nu_in[i], v = nu_in[n + i], r = nu_in[2 * n + i];
  } else {
    sample_reset(p.seed, p.env_off + i, epi, p.reset_scale, N, E, psi, u, v, r);
  }
  p.eta[i] = N, p.eta[n + i] = E, p.eta[2 * n + i] = psi;
  p.nu[i] = u, p.nu[n + i] = v, p.nu[2 * n + i] = r;
  float rN, rE, rP;                                                                    // what obs rows 0-2 are formed against
  if (rf.state != nullptr) {                                                           // reference model attached
    rN = N, rE = E, rP = psi;
    rf.state[i] = N, rf.state[n + i] = E, rf.state[2 * n + i] = psi;
#pragma unroll
    for (int q = 3; q < 9; ++q) rf.state[q * n + i] = 0.f;
  } else {
    rN = p.ref[i], rE = p.ref[n + i], rP = p.ref[2 * n + i];
  }
  float t0[3] = {0.f, 0.f, 0.f};                                                       // customEnv.py:190
  if (p.reset_acts) sample_reset_thrust(p.seed, p.env_off + i, epi, t0);               // :179-188
  p.prev_thrust[i] = t0[0], p.prev_thrust[n + i] = t0[1], p.prev_thrust[2 * n + i] = t0[2];
  p.angles[i] = T::DEF_BOW, p.angles[n + i] = T::DEF_PORT, p.angles[2 * n + i] = T::DEF_STAR;  // :173-177,192
  p.tau_act[i] = 0.f, p.tau_act[n + i] = 0.f, p.tau_act[2 * n + i] = 0.f;
  p.obs_tail[i] = div100(t0[0]), p.obs_tail[n + i] = div100(t0[1]), p.obs_tail[2 * n + i] = div100(t0[2]);
  if (d.current != nullptr) {                                                          // disturbance enabled
    float cur[2], b[3];
    sample_disturbance(p.seed, p.env_off + i, epi, d.k, cur, b);
    d.current[i] = cur[0], d.current[n + i] = cur[1];
    d.bias[i] = b[0], d.bias[n + i] = b[1], d.bias[2 * n + i] = b[2];
  }
  if (wv.motion != nullptr) {                                                        // waves enabled
    float x[3], xd[3], w0;
    sample_waves(p.seed, p.env_off + i, epi, wv.k.sigma[0], wv.k.sigma[1], wv.k.sigma[2], wv.k.omega_lo, wv.k.omega_span,
                 x, xd, &w0);
#pragma unroll
    for (int c = 0; c < 3; ++c) wv.motion[c * n + i] = x[c], wv.rate[c * n + i] = xd[c];
    wv.omega[i] = w0;
    add_wave_motion(N, E, psi, u, v, r, x, xd);                                        // the observation is measured
  }
  if (ob.state != nullptr) {                                                           // observer attached
    float x[15];
    const float y[3] = {N, E, psi};
    observer_reset_column(x, y);
#pragma unroll
    for (int c = 0; c < 15; ++c) ob.state[c * n + i] = x[c];
    u = v = r = 0.f;                                                                   // nu^ of the observation
  }
  p.ep_len[i] = next_episode_word(epi);
  if (obs != nullptr) {
    float xb, yb, pb;
    error_frame(N, E, psi, rN, rE, rP, xb, yb, pb);
    obs[i] = xb, obs[n + i] = yb, obs[2 * n + i] = pb;
    obs[3 * n + i] = u, obs[4 * n + i] = v, obs[5 * n + i] = r;
    if constexpr (EXT) obs[6 * n + i] = div100(t0[0]), obs[7 * n + i] = div100(t0[1]), obs[8 * n + i] = div100(t0[2]);
  }
}

}  // namespace ml4ca
