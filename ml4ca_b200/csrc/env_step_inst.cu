// env_step_inst.cu -- one translation unit per env class (compiled with -DML4CA_STEP_UNIT=0..4) so that the
// kernel instantiations of env_kernels.cuh build in parallel.  Units: 0 full, 1 simple, 2 limited,
// 3 final (wrapped angles), 4 final (continuous angles).
#include <stdlib.h>

#include "env_kernels.cuh"

#ifndef ML4CA_STEP_UNIT
#error "compile with -DML4CA_STEP_UNIT=<0..4>"
#endif

namespace ml4ca {

#if ML4CA_STEP_UNIT == 0
#define UNIT_KIND ML4CA_ENV_FULL
#define UNIT_CONT false
#define UNIT_NAME launch_step_full
#define UNIT_RESET launch_reset_full
#elif ML4CA_STEP_UNIT == 1
#define UNIT_KIND ML4CA_ENV_SIMPLE
#define UNIT_CONT false
#define UNIT_NAME launch_step_simple
#define UNIT_RESET launch_reset_simple
#elif ML4CA_STEP_UNIT == 2
#define UNIT_KIND ML4CA_ENV_LIMITED
#define UNIT_CONT false
#define UNIT_NAME launch_step_limited
#define UNIT_RESET launch_reset_limited
#elif ML4CA_STEP_UNIT == 3
#define UNIT_KIND ML4CA_ENV_FINAL
#define UNIT_CONT false
#define UNIT_NAME launch_step_final_wrap
#define UNIT_RESET launch_reset_final_wrap
#else
#define UNIT_KIND ML4CA_ENV_FINAL
#define UNIT_CONT true
#define UNIT_NAME launch_step_final_cont
#define UNIT_RESET launch_reset_final_cont
#endif

// The scalar kernels with the reference model in the loop, with or without the observer (OBSV), any LAG / DIST / WAVE.
template <int KIND, bool CONT, bool EXT, bool OBSV>
static void launch_step_ref(bool lag, bool dist, bool wave, unsigned blocks, const EnvParams& p, const DistParams& d,
                            const WaveParams& w, const ObserverParams& ob, const RefParams& rf, const float* action,
                            float* obs, float* rew, uint8_t* done, cudaStream_t st) {
#define ML4CA_REF(L, D, W) \
  env_step_kernel<KIND, CONT, EXT, 1, L, D, W, OBSV, true><<<blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf)
  if (wave) {
    if (lag && dist) ML4CA_REF(true, true, true);
    else if (lag) ML4CA_REF(true, false, true);
    else if (dist) ML4CA_REF(false, true, true);
    else ML4CA_REF(false, false, true);
  } else {
    if (lag && dist) ML4CA_REF(true, true, false);
    else if (lag) ML4CA_REF(true, false, false);
    else if (dist) ML4CA_REF(false, true, false);
    else ML4CA_REF(false, false, false);
  }
#undef ML4CA_REF
}

template <int KIND, bool CONT, bool EXT>
static int launch_step_vec(const ml4ca_env* e, const EnvParams& p, const DistParams& d, const WaveParams& w,
                           const ObserverParams& ob, const RefParams& rf, const float* action, float* obs, float* rew,
                           uint8_t* done, cudaStream_t st) {
  const int64_t n = p.count;
  if (rf.state != nullptr) {      // reference model attached: the scalar kernel with the model (and the observer) in the loop
    const unsigned blocks = (unsigned)((n + 255) / 256);
    const bool lag = e->cfg.actuator_lag_s > 0.f, dist = d.current != nullptr, wave = w.motion != nullptr;
    if (ob.state != nullptr)
      launch_step_ref<KIND, CONT, EXT, true>(lag, dist, wave, blocks, p, d, w, ob, rf, action, obs, rew, done, st);
    else
      launch_step_ref<KIND, CONT, EXT, false>(lag, dist, wave, blocks, p, d, w, ob, rf, action, obs, rew, done, st);
    return check_launch("env_step_kernel<ref>");
  }
  if (ob.state != nullptr) {      // observer attached: the scalar kernel with the observer in the loop, any LAG / DIST / WAVE
    const unsigned blocks = (unsigned)((n + 255) / 256);
    const bool lag = e->cfg.actuator_lag_s > 0.f, dist = d.current != nullptr, wave = w.motion != nullptr;
#define ML4CA_OBSV(L, D, W) \
  env_step_kernel<KIND, CONT, EXT, 1, L, D, W, true><<<blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf)
    if (wave) {
      if (lag && dist) ML4CA_OBSV(true, true, true);
      else if (lag) ML4CA_OBSV(true, false, true);
      else if (dist) ML4CA_OBSV(false, true, true);
      else ML4CA_OBSV(false, false, true);
    } else {
      if (lag && dist) ML4CA_OBSV(true, true, false);
      else if (lag) ML4CA_OBSV(true, false, false);
      else if (dist) ML4CA_OBSV(false, true, false);
      else ML4CA_OBSV(false, false, false);
    }
#undef ML4CA_OBSV
    return check_launch("env_step_kernel<obsv>");
  }
  if (w.motion != nullptr) {      // waves enabled: the scalar kernel with seven more state rows (and the disturbance's)
    const int64_t blocks = (n + 255) / 256;
    const bool lag = e->cfg.actuator_lag_s > 0.f, dist = d.current != nullptr;
    if (lag && dist)
      env_step_kernel<KIND, CONT, EXT, 1, true, true, true><<<(unsigned)blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
    else if (lag)
      env_step_kernel<KIND, CONT, EXT, 1, true, false, true><<<(unsigned)blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
    else if (dist)
      env_step_kernel<KIND, CONT, EXT, 1, false, true, true><<<(unsigned)blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
    else
      env_step_kernel<KIND, CONT, EXT, 1, false, false, true><<<(unsigned)blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
    return check_launch("env_step_kernel<wave>");
  }
  if (d.current != nullptr) {          // disturbance enabled: the scalar kernel with five more state rows
    const int64_t blocks = (n + 255) / 256;
    if (e->cfg.actuator_lag_s > 0.f)
      env_step_kernel<KIND, CONT, EXT, 1, true, true><<<(unsigned)blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
    else
      env_step_kernel<KIND, CONT, EXT, 1, false, true><<<(unsigned)blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
    return check_launch("env_step_kernel<dist>");
  }
  if (e->cfg.actuator_lag_s > 0.f) {   // lagged wrench: the scalar kernel with three more state rows
    const int64_t blocks = (n + 255) / 256;
    env_step_kernel<KIND, CONT, EXT, 1, true><<<(unsigned)blocks, 256, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
    return check_launch("env_step_kernel<lag>");
  }
  const bool vec4 = (p.n % 4 == 0) && (n % 4 == 0) && (p.io_stride % 4 == 0) && aligned16(p.eta) && aligned16(action) &&
                    aligned16(obs) && aligned16(rew) && ((reinterpret_cast<uintptr_t>(done) & 3u) == 0);
  static const int threads = [] {   // tuning knob: ML4CA_ENV_THREADS=64|128|256
    const char* e = getenv("ML4CA_ENV_THREADS");
    const int t = e ? atoi(e) : 256;
    return (t == 64 || t == 128 || t == 256) ? t : 256;
  }();
  // Two envs per thread is the default: the kernel is issue-bound, and the packed-FP32 integrator (FFMA2) of the
  // two-env variant issues 28 % fewer instructions per env-step than the scalar one (profiles/env_step_r1.md:
  // 0.50 ms vs 0.59 ms for 16 Mi envs).  One env per thread serves batches whose rows are not 16-byte aligned.
  static const int vec_pref = [] {   // tuning knob: ML4CA_ENV_VEC=1|2|4
    const char* e = getenv("ML4CA_ENV_VEC");
    return e ? atoi(e) : 2;
  }();
  const int vec = (vec4 && (vec_pref == 4 || vec_pref == 2)) ? vec_pref : 1;
  if (vec == 4) {
    const int64_t blocks = (n / 4 + threads - 1) / threads;
    env_step_kernel<KIND, CONT, EXT, 4><<<(unsigned)blocks, threads, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
  } else if (vec == 2) {
    const int64_t blocks = (n / 2 + threads - 1) / threads;
    env_step_kernel<KIND, CONT, EXT, 2><<<(unsigned)blocks, threads, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
  } else {
    const int64_t blocks = (n + threads - 1) / threads;
    env_step_kernel<KIND, CONT, EXT, 1><<<(unsigned)blocks, threads, 0, st>>>(p, action, obs, rew, done, d, w, ob, rf);
  }
  return check_launch("env_step_kernel");
}

int UNIT_NAME(const ml4ca_env* e, const EnvParams& p, const DistParams& d, const WaveParams& w, const ObserverParams& ob,
              const RefParams& rf, const float* action, float* obs, float* rew, uint8_t* done, cudaStream_t st) {
  if (e->cfg.extended_state) {
#if ML4CA_STEP_UNIT == 1
    return ML4CA_ERR_UNSUPPORTED;
#else
    return launch_step_vec<UNIT_KIND, UNIT_CONT, true>(e, p, d, w, ob, rf, action, obs, rew, done, st);
#endif
  }
  return launch_step_vec<UNIT_KIND, UNIT_CONT, false>(e, p, d, w, ob, rf, action, obs, rew, done, st);
}

int UNIT_RESET(const ml4ca_env* e, const EnvParams& p, const uint8_t* mask, const float* eta, const float* nu,
               float* obs, cudaStream_t st) {
  const DistParams& d = e->dist;
  const WaveParams& w = e->wave;
  const int threads = 256;
  const int64_t blocks = (e->n + threads - 1) / threads;
  if (e->cfg.extended_state)
    env_reset_kernel<UNIT_KIND, UNIT_CONT, true><<<(unsigned)blocks, threads, 0, st>>>(p, mask, eta, nu, obs, d, w, e->obsv, e->refm);
  else
    env_reset_kernel<UNIT_KIND, UNIT_CONT, false><<<(unsigned)blocks, threads, 0, st>>>(p, mask, eta, nu, obs, d, w, e->obsv, e->refm);
  return check_launch("env_reset_kernel");
}

}  // namespace ml4ca
