// env_step.cu -- host side of K3: handle life cycle and the extern "C" entry points of the env.
// Kernels: env_kernels.cuh; per-class instantiations: env_step_inst.cu.
#include <stdlib.h>

#include <cmath>
#include <new>

#include "env_kernels.cuh"

namespace ml4ca {

__global__ void __launch_bounds__(256) error_frame_kernel(int64_t n, const float* __restrict__ eta,
                                                          const float* __restrict__ ref, float* __restrict__ err) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float xb, yb, pb;
  error_frame(eta[i], eta[n + i], eta[2 * n + i], ref[i], ref[n + i], ref[2 * n + i], xb, yb, pb);
  err[i] = xb, err[n + i] = yb, err[2 * n + i] = pb;
}

// Revolt.state() / state_extended() (customEnv.py:196-205) from the state in HBM; with waves enabled, of the measured
// pose and velocity; with an observer attached, rows 0-5 of its estimates eta^ and nu^; with a reference model attached,
// rows 0-2 against its eta_d.
__global__ void __launch_bounds__(256) observe_kernel(const EnvParams p, int ext, float* __restrict__ obs,
                                                      const WaveParams w, const ObserverParams ob, const RefParams rf) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = p.n;
  if (i >= n) return;
  float N = p.eta[i], E = p.eta[n + i], psi = p.eta[2 * n + i], u = p.nu[i], v = p.nu[n + i], r = p.nu[2 * n + i];
  if (w.motion != nullptr) {
    const float x[3] = {w.motion[i], w.motion[n + i], w.motion[2 * n + i]};
    const float xd[3] = {w.rate[i], w.rate[n + i], w.rate[2 * n + i]};
    add_wave_motion(N, E, psi, u, v, r, x, xd);
  }
  if (ob.state != nullptr) {
    N = ob.state[6 * n + i], E = ob.state[7 * n + i], psi = ob.state[8 * n + i];
    u = ob.state[9 * n + i], v = ob.state[10 * n + i], r = ob.state[11 * n + i];
  }
  const float* ref = rf.state != nullptr ? rf.state : p.ref;                        // eta_d: rows 0-2 of the model's state
  float xb, yb, pb;
  error_frame(N, E, psi, ref[i], ref[n + i], ref[2 * n + i], xb, yb, pb);
  obs[i] = xb, obs[n + i] = yb, obs[2 * n + i] = pb;
  obs[3 * n + i] = u, obs[4 * n + i] = v, obs[5 * n + i] = r;
  if (ext) obs[6 * n + i] = p.obs_tail[i], obs[7 * n + i] = p.obs_tail[n + i], obs[8 * n + i] = p.obs_tail[2 * n + i];
}

__global__ void __launch_bounds__(256) unpack_ep_len_kernel(int64_t n, const int32_t* __restrict__ word,
                                                            int32_t* __restrict__ ep_len) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) ep_len[i] = (int32_t)((uint32_t)word[i] & kEpLenMask);
}

template <int KIND, bool CONT>
__global__ void __launch_bounds__(256) scale_clip_kernel(int64_t n, const float* __restrict__ action,
                                                         float* __restrict__ act_env, int8_t* __restrict__ sat_out) {
  using T = EnvTraits<KIND, CONT>;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float a[T::ACT], cmd[T::NCMD];
  int sat[T::NCMD];
#pragma unroll
  for (int c = 0; c < T::ACT; ++c) a[c] = action[(int64_t)c * n + i];
  transform_action<KIND, CONT>(a, cmd, sat);
#pragma unroll
  for (int c = 0; c < T::NCMD; ++c) {
    act_env[(int64_t)c * n + i] = cmd[c];
    if (sat_out != nullptr) sat_out[(int64_t)c * n + i] = (int8_t)sat[c];
  }
}

// ---- host-side dispatch -------------------------------------------------------------------------------------------
static int validate_cfg(const ml4ca_env_cfg* c) {
  ML4CA_REQUIRE(c != nullptr, "cfg is NULL");
  ML4CA_REQUIRE(c->kind >= ML4CA_ENV_FULL && c->kind <= ML4CA_ENV_FINAL, "unknown env kind");
  ML4CA_REQUIRE(!(c->cont_ang && c->kind != ML4CA_ENV_FINAL),
                "continuous angles only work with the final environment (customEnv.py:228)");
  ML4CA_REQUIRE(!(c->kind == ML4CA_ENV_SIMPLE && c->extended_state),
                "RevoltSimple has no azimuth bound for the extended-state penalty (customEnv.py:319,339)");
  ML4CA_REQUIRE(c->n_substeps >= 0 && c->max_ep_len > 0 && c->max_ep_len <= 65535,
                "n_substeps >= 0 and 0 < max_ep_len <= 65535 required");
  ML4CA_REQUIRE(c->hull_model == 0 || c->hull_model == 1, "hull_model must be 0 (default constants) or 1 (box-test fit)");
  ML4CA_REQUIRE(c->actuator_lag_s >= 0.f && c->actuator_lag_s <= 60.f, "actuator_lag_s must lie in [0, 60] s");
  return ML4CA_OK;
}

static int validate_disturbance(const ml4ca_disturbance_cfg* d) {
  ML4CA_REQUIRE(std::isfinite(d->current_speed_min) && std::isfinite(d->current_speed_max) &&
                    std::isfinite(d->current_dir_min) && std::isfinite(d->current_dir_max) &&
                    std::isfinite(d->bias_time_s) && std::isfinite(d->bias_std[0]) && std::isfinite(d->bias_std[1]) &&
                    std::isfinite(d->bias_std[2]),
                "disturbance: every field must be finite");
  ML4CA_REQUIRE(d->current_speed_min >= 0.f && d->current_speed_min <= d->current_speed_max,
                "disturbance: current speed range needs 0 <= current_speed_min <= current_speed_max");
  ML4CA_REQUIRE(d->current_dir_min <= d->current_dir_max, "disturbance: current direction range needs current_dir_min <= current_dir_max");
  ML4CA_REQUIRE(d->bias_std[0] >= 0.f && d->bias_std[1] >= 0.f && d->bias_std[2] >= 0.f,
                "disturbance: bias_std must be non-negative");
  ML4CA_REQUIRE(d->bias_time_s >= 0.f, "disturbance: bias_time_s must be non-negative (0 = constant over the episode)");
  return ML4CA_OK;
}

// Per-launch constants of the disturbance (env_math.cuh: DistConsts).
static DistConsts dist_consts(const ml4ca_env_cfg& c, const ml4ca_disturbance_cfg& d) {
  DistConsts k;
  k.speed_lo = d.current_speed_min;
  k.speed_span = d.current_speed_max - d.current_speed_min;
  k.dir_lo = d.current_dir_min;
  k.dir_span = d.current_dir_max - d.current_dir_min;
  const double a = d.bias_time_s > 0.f ? std::exp(-(double)c.step_dt / (double)d.bias_time_s) : 1.0;
  k.gm_a = (float)a;
  for (int i = 0; i < 3; ++i) {
    k.bias_std[i] = d.bias_std[i];
    k.gm_gain[i] = (float)((double)d.bias_std[i] * std::sqrt(1.0 - a * a));
  }
  k.t_step = (float)((double)c.n_substeps * (double)c.sim_dt);
  k.gm = d.bias_time_s > 0.f ? 1 : 0;
  k.noise = (k.gm && (d.bias_std[0] > 0.f || d.bias_std[1] > 0.f || d.bias_std[2] > 0.f)) ? 1 : 0;
  return k;
}

// The disturbance state of every env, drawn as a reset would draw it (episode word of the moment).
__global__ void __launch_bounds__(256) draw_disturbance_kernel(const EnvParams p, const DistParams d) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = p.n;
  if (i >= n) return;
  float cur[2], b[3];
  sample_disturbance(p.seed, p.env_off + i, p.ep_len[i], d.k, cur, b);
  d.current[i] = cur[0], d.current[n + i] = cur[1];
  d.bias[i] = b[0], d.bias[n + i] = b[1], d.bias[2 * n + i] = b[2];
}

static int validate_waves(const ml4ca_env_cfg& c, const ml4ca_wave_cfg* w) {
  ML4CA_REQUIRE(std::isfinite(w->sigma[0]) && std::isfinite(w->sigma[1]) && std::isfinite(w->sigma[2]) &&
                    std::isfinite(w->omega_min) && std::isfinite(w->omega_max) && std::isfinite(w->damping),
                "waves: every field must be finite");
  ML4CA_REQUIRE(w->sigma[0] >= 0.f && w->sigma[1] >= 0.f && w->sigma[2] >= 0.f, "waves: sigma must be non-negative");
  ML4CA_REQUIRE(w->omega_min > 0.f && w->omega_min <= w->omega_max,
                "waves: peak frequency range needs 0 < omega_min <= omega_max");
  ML4CA_REQUIRE((double)w->omega_max * (double)c.step_dt < ML4CA_PI,
                "waves: omega_max * step_dt must stay below pi (the observation would alias the motion)");
  ML4CA_REQUIRE(w->damping > 0.f && w->damping < 1.f, "waves: damping must lie in (0, 1)");
  return ML4CA_OK;
}

// Per-launch constants of the wave motion (env_math.cuh: WaveConsts).
static WaveConsts wave_consts(const ml4ca_env_cfg& c, const ml4ca_wave_cfg& w) {
  WaveConsts k;
  const double lam = w.damping, sq = std::sqrt(1.0 - lam * lam), dt = c.step_dt;
  for (int i = 0; i < 3; ++i) k.sigma[i] = w.sigma[i];
  k.omega_lo = w.omega_min;
  k.omega_span = w.omega_max - w.omega_min;
  k.lam_dt = (float)(lam * dt);
  k.wd_dt = (float)(sq * dt);
  k.lam_ratio = (float)(lam / sq);
  k.inv_sq = (float)(1.0 / sq);
  k.noise = (w.sigma[0] > 0.f || w.sigma[1] > 0.f || w.sigma[2] > 0.f) ? 1 : 0;
  return k;
}

// The wave state of every env, drawn as a reset would draw it (episode word of the moment).
__global__ void __launch_bounds__(256) draw_waves_kernel(const EnvParams p, const WaveParams w) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = p.n;
  if (i >= n) return;
  float x[3], xd[3], w0;
  sample_waves(p.seed, p.env_off + i, p.ep_len[i], w.k.sigma[0], w.k.sigma[1], w.k.sigma[2], w.k.omega_lo, w.k.omega_span, x,
               xd, &w0);
#pragma unroll
  for (int c = 0; c < 3; ++c) w.motion[c * n + i] = x[c], w.rate[c * n + i] = xd[c];
  w.omega[i] = w0;
}

// ml4ca_env_set_observer: every env's observer column starts from its current measured pose (eta^ = y, the rest 0).
__global__ void __launch_bounds__(256) attach_observer_kernel(const EnvParams p, const WaveParams w, const ObserverParams ob) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = p.n;
  if (i >= n) return;
  float N = p.eta[i], E = p.eta[n + i], psi = p.eta[2 * n + i], u = 0.f, v = 0.f, r = 0.f;
  if (w.motion != nullptr) {
    const float x[3] = {w.motion[i], w.motion[n + i], w.motion[2 * n + i]};
    const float xd[3] = {0.f, 0.f, 0.f};
    add_wave_motion(N, E, psi, u, v, r, x, xd);
  }
  float s[15];
  const float y[3] = {N, E, psi};
  observer_reset_column(s, y);
#pragma unroll
  for (int c = 0; c < 15; ++c) ob.state[c * n + i] = s[c];
}

// ml4ca_env_set_refmodel: every env's reference-model column starts from its current LF pose (eta_d = eta, v_d = a_d = 0).
__global__ void __launch_bounds__(256) attach_refmodel_kernel(const EnvParams p, const RefParams rf) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = p.n;
  if (i >= n) return;
#pragma unroll
  for (int c = 0; c < 3; ++c) rf.state[c * n + i] = p.eta[c * n + i];
#pragma unroll
  for (int q = 3; q < 9; ++q) rf.state[q * n + i] = 0.f;
}

static void make_reset_scale(const ml4ca_env_cfg& c, float fraction, float (&scale)[6]) {
  // fp32, one rounding per product, same order as oracle/env_oracle.py::sample_reset
  const float vfr = (float)ML4CA_VEL_FRACTION * fraction;
  for (int i = 0; i < 3; ++i) scale[i] = c.ss_bounds[i] * fraction;
  for (int i = 3; i < 6; ++i) scale[i] = c.ss_bounds[i] * vfr;
}

#define ML4CA_DECL_UNIT(name)                                                                                   \
  int launch_step_##name(const ml4ca_env*, const EnvParams&, const DistParams&, const WaveParams&,              \
                         const ObserverParams&, const RefParams&, const float*, float*, float*, uint8_t*,       \
                         cudaStream_t);                                                                         \
  int launch_reset_##name(const ml4ca_env*, const EnvParams&, const uint8_t*, const float*, const float*, float*, \
                          cudaStream_t);
ML4CA_DECL_UNIT(full)
ML4CA_DECL_UNIT(simple)
ML4CA_DECL_UNIT(limited)
ML4CA_DECL_UNIT(final_wrap)
ML4CA_DECL_UNIT(final_cont)
#undef ML4CA_DECL_UNIT

// Step the slice [first, first + count) of the batch; action / obs rows have stride io_stride.
static int launch_step(const ml4ca_env* e, int64_t first, int64_t count, int64_t io_stride, const float* action,
                       float* obs, float* rew, uint8_t* done, cudaStream_t st) {
  EnvParams p = e->p;
  p.eta += first, p.nu += first, p.ref += first, p.prev_thrust += first, p.angles += first, p.obs_tail += first;
  p.tau_act += first;
  p.ep_len += first;
  if (p.cut_obs != nullptr) p.cut_obs += first;
  DistParams d = e->dist;
  if (d.current != nullptr) d.current += first, d.bias += first;
  WaveParams w = e->wave;
  if (w.motion != nullptr) w.motion += first, w.rate += first, w.omega += first;
  ObserverParams ob = e->obsv;
  if (ob.state != nullptr) ob.state += first, ob.omega += first;
  RefParams rf = e->refm;
  if (rf.state != nullptr) rf.state += first;
  p.env_off += first;
  p.count = count;
  p.io_stride = io_stride;
  switch (e->cfg.kind) {
    case ML4CA_ENV_FULL: return launch_step_full(e, p, d, w, ob, rf, action, obs, rew, done, st);
    case ML4CA_ENV_SIMPLE: return launch_step_simple(e, p, d, w, ob, rf, action, obs, rew, done, st);
    case ML4CA_ENV_LIMITED: return launch_step_limited(e, p, d, w, ob, rf, action, obs, rew, done, st);
    default:
      return e->cfg.cont_ang ? launch_step_final_cont(e, p, d, w, ob, rf, action, obs, rew, done, st)
                             : launch_step_final_wrap(e, p, d, w, ob, rf, action, obs, rew, done, st);
  }
}

static int launch_reset(const ml4ca_env* e, const EnvParams& p, const uint8_t* mask, const float* eta,
                        const float* nu, float* obs, cudaStream_t st) {
  switch (e->cfg.kind) {
    case ML4CA_ENV_FULL: return launch_reset_full(e, p, mask, eta, nu, obs, st);
    case ML4CA_ENV_SIMPLE: return launch_reset_simple(e, p, mask, eta, nu, obs, st);
    case ML4CA_ENV_LIMITED: return launch_reset_limited(e, p, mask, eta, nu, obs, st);
    default:
      return e->cfg.cont_ang ? launch_reset_final_cont(e, p, mask, eta, nu, obs, st)
                             : launch_reset_final_wrap(e, p, mask, eta, nu, obs, st);
  }
}

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) ok = false;
    if (ok && prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

}  // namespace ml4ca

using namespace ml4ca;

extern "C" {

int ml4ca_env_cfg_default(int32_t kind, int32_t cont_ang, int32_t extended_state, ml4ca_env_cfg* out) {
  ML4CA_REQUIRE(out != nullptr, "out is NULL");
  ml4ca_env_cfg c = {};
  c.kind = kind;
  c.cont_ang = cont_ang ? 1 : 0;
  c.extended_state = extended_state ? 1 : 0;
  c.n_substeps = ML4CA_N_SUBSTEPS;
  c.max_ep_len = ML4CA_MAX_EP_LEN;  // int(800 * 10 / 20), customEnv.py:83
  c.auto_reset = 0;
  const float b_full[6] = {8.0f, 8.0f, (float)(ML4CA_PI / 2), 1.4f, 0.30f, 0.52f};    // customEnv.py:26
  const float b_simple[6] = {8.0f, 8.0f, (float)(ML4CA_PI / 2), 1.75f, 0.30f, 0.51f};  // :337
  for (int i = 0; i < 6; ++i) c.ss_bounds[i] = (kind == ML4CA_ENV_SIMPLE) ? b_simple[i] : b_full[i];
  if (kind == ML4CA_ENV_LIMITED || kind == ML4CA_ENV_FINAL) c.ss_bounds[2] = (float)ML4CA_BOUND_YAW;  // :361,386
  c.sim_dt = (float)ML4CA_SIM_DT;
  c.step_dt = (float)(0.01 * ML4CA_N_SUBSTEPS);
  c.reset_fraction = 0.8f;
  c.seed = 0;
  c.env_id_offset = 0;
  int st = validate_cfg(&c);
  if (st != ML4CA_OK) return st;
  *out = c;
  return ML4CA_OK;
}

int ml4ca_env_dims(const ml4ca_env_cfg* cfg, int32_t* act_dim, int32_t* obs_dim) {
  int st = validate_cfg(cfg);
  if (st != ML4CA_OK) return st;
  static const int act[4] = {6, 3, 5, 5};
  if (act_dim) *act_dim = (cfg->kind == ML4CA_ENV_FINAL && cfg->cont_ang) ? 7 : act[cfg->kind];
  if (obs_dim) *obs_dim = cfg->extended_state ? 9 : 6;
  return ML4CA_OK;
}

int ml4ca_env_create(const ml4ca_env_cfg* cfg, int64_t n_env, int32_t device, ml4ca_env** out) {
  ML4CA_REQUIRE(out != nullptr, "out is NULL");
  *out = nullptr;
  int st = validate_cfg(cfg);
  if (st != ML4CA_OK) return st;
  ML4CA_REQUIRE(n_env > 0, "n_env must be positive");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("ml4ca_env_create: no CUDA device (this library has no CPU fallback)");
    return ML4CA_ERR_NO_DEVICE;
  }
  ML4CA_REQUIRE(device >= 0 && device < ndev, "device index out of range");
  DeviceGuard guard(device);
  ml4ca_env* e = new (std::nothrow) ml4ca_env();
  ML4CA_REQUIRE(e != nullptr, "out of host memory");
  e->cfg = *cfg;
  e->n = n_env;
  e->device = device;
  e->tail_valid = true;
  // one slab: 21 fp32 rows + 1 int32 row (the episode words), each row padded to a 16-byte multiple so that every row start is
  // float4-aligned whenever n % 4 == 0 (rows are indexed with stride n, so the padding only sits at the end).
  const size_t row = (size_t)n_env * sizeof(float);
  const size_t bytes = 22 * row + 256;
  cudaError_t ce = cudaMalloc(&e->slab, bytes);
  if (ce != cudaSuccess) {
    delete e;
    return check_cuda(ce, "cudaMalloc(env state)");
  }
  ce = cudaMemset(e->slab, 0, bytes);
  if (ce != cudaSuccess) {
    cudaFree(e->slab);
    delete e;
    return check_cuda(ce, "cudaMemset(env state)");
  }
  float* f = static_cast<float*>(e->slab);
  EnvParams& p = e->p;
  p.eta = f;
  p.nu = f + 3 * n_env;
  p.ref = f + 6 * n_env;
  p.prev_thrust = f + 9 * n_env;
  p.angles = f + 12 * n_env;
  p.obs_tail = f + 15 * n_env;
  p.tau_act = f + 18 * n_env;
  p.ep_len = reinterpret_cast<int32_t*>(f + 21 * n_env);
  p.cut_obs = nullptr;
  p.n = n_env;
  for (int i = 0; i < 6; ++i) p.bounds[i] = cfg->ss_bounds[i];
  make_reset_scale(*cfg, cfg->reset_fraction, p.reset_scale);
  p.inv_step_dt = 1.0f / cfg->step_dt;
  p.pad1 = 0.f;
  p.hull = hull_consts(cfg->sim_dt, cfg->hull_model, cfg->actuator_lag_s);
  p.n_sub = cfg->n_substeps;
  p.max_ep_len = cfg->max_ep_len;
  p.auto_reset = cfg->auto_reset;
  p.reset_acts = cfg->reset_acts ? 1 : 0;
  p.seed = cfg->seed;
  p.env_off = cfg->env_id_offset;
  p.count = n_env;
  p.io_stride = n_env;
  *out = e;
  return ML4CA_OK;
}

int ml4ca_env_destroy(ml4ca_env* env) {
  if (env == nullptr) return ML4CA_OK;
  DeviceGuard guard(env->device);
  if (env->pipe != nullptr) {
    HostPipe* hp = env->pipe;
    cudaStreamSynchronize(hp->s_out);
    cudaStreamDestroy(hp->s_in), cudaStreamDestroy(hp->s_k), cudaStreamDestroy(hp->s_out);
    cudaEventDestroy(hp->ev_start);
    for (int s = 0; s < 2; ++s) cudaEventDestroy(hp->ev_in[s]), cudaEventDestroy(hp->ev_k[s]), cudaEventDestroy(hp->ev_out[s]);
    cudaFree(hp->slab);
    delete hp;
  }
  cudaFree(env->dist_slab);
  cudaFree(env->wave_slab);
  cudaFree(env->slab);
  delete env;
  return ML4CA_OK;
}

int64_t ml4ca_env_size(const ml4ca_env* env) { return env ? env->n : 0; }

int ml4ca_env_reset(ml4ca_env* env, const uint8_t* mask, float fraction, float* obs, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  DeviceGuard guard(env->device);
  EnvParams p = env->p;
  make_reset_scale(env->cfg, fraction, p.reset_scale);
  if (mask == nullptr) env->tail_valid = true;
  return launch_reset(env, p, mask, nullptr, nullptr, obs, static_cast<cudaStream_t>(stream));
}

int ml4ca_env_reset_to(ml4ca_env* env, const uint8_t* mask, const float* eta, const float* nu, float* obs,
                       void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  ML4CA_REQUIRE(eta != nullptr && nu != nullptr, "eta and nu are required");
  DeviceGuard guard(env->device);
  if (mask == nullptr) env->tail_valid = true;
  return launch_reset(env, env->p, mask, eta, nu, obs, static_cast<cudaStream_t>(stream));
}

int ml4ca_env_set_cut_obs(ml4ca_env* env, float* cut_obs) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  env->p.cut_obs = cut_obs;
  return ML4CA_OK;
}

int ml4ca_env_set_reset_fraction(ml4ca_env* env, float fraction) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  ML4CA_REQUIRE(fraction >= 0.f, "fraction must be non-negative");
  env->cfg.reset_fraction = fraction;
  make_reset_scale(env->cfg, fraction, env->p.reset_scale);
  return ML4CA_OK;
}

int ml4ca_env_set_disturbance(ml4ca_env* env, const ml4ca_disturbance_cfg* cfg, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  if (cfg == nullptr) {
    env->dist.current = env->dist.bias = nullptr;     // the rows stay allocated for a later enable
    return ML4CA_OK;
  }
  int stv = validate_disturbance(cfg);
  if (stv != ML4CA_OK) return stv;
  DeviceGuard guard(env->device);
  const int64_t n = env->n;
  if (env->dist_slab == nullptr) ML4CA_CUDA(cudaMalloc(&env->dist_slab, 5 * (size_t)n * sizeof(float) + 256));
  float* f = static_cast<float*>(env->dist_slab);
  env->dist.current = f;
  env->dist.bias = f + 2 * n;
  env->dist.k = dist_consts(env->cfg, *cfg);
  draw_disturbance_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(env->p, env->dist);
  return check_launch("draw_disturbance_kernel");
}

int ml4ca_env_set_disturbance_state(ml4ca_env* env, const float* current, const float* bias, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  ML4CA_REQUIRE(env->dist.current != nullptr, "no disturbance is enabled (ml4ca_env_set_disturbance)");
  DeviceGuard guard(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t row = (size_t)env->n * sizeof(float);
  if (current) ML4CA_CUDA(cudaMemcpyAsync(env->dist.current, current, 2 * row, cudaMemcpyDeviceToDevice, st));
  if (bias) ML4CA_CUDA(cudaMemcpyAsync(env->dist.bias, bias, 3 * row, cudaMemcpyDeviceToDevice, st));
  return ML4CA_OK;
}

int ml4ca_env_get_disturbance(ml4ca_env* env, float* current, float* bias, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  ML4CA_REQUIRE(env->dist.current != nullptr, "no disturbance is enabled (ml4ca_env_set_disturbance)");
  DeviceGuard guard(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t row = (size_t)env->n * sizeof(float);
  if (current) ML4CA_CUDA(cudaMemcpyAsync(current, env->dist.current, 2 * row, cudaMemcpyDeviceToDevice, st));
  if (bias) ML4CA_CUDA(cudaMemcpyAsync(bias, env->dist.bias, 3 * row, cudaMemcpyDeviceToDevice, st));
  return ML4CA_OK;
}

int ml4ca_env_set_waves(ml4ca_env* env, const ml4ca_wave_cfg* cfg, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  WaveParams& w = env->wave;
  if (cfg == nullptr) {
    w.motion = w.rate = w.omega = nullptr;            // the rows stay allocated for a later enable
    return ML4CA_OK;
  }
  int stv = validate_waves(env->cfg, cfg);
  if (stv != ML4CA_OK) return stv;
  DeviceGuard guard(env->device);
  const int64_t n = env->n;
  if (env->wave_slab == nullptr) ML4CA_CUDA(cudaMalloc(&env->wave_slab, 7 * (size_t)n * sizeof(float) + 256));
  float* f = static_cast<float*>(env->wave_slab);
  w.motion = f;
  w.rate = f + 3 * n;
  w.omega = f + 6 * n;
  w.k = wave_consts(env->cfg, *cfg);
  draw_waves_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(env->p, w);
  return check_launch("draw_waves_kernel");
}

int ml4ca_env_set_wave_state(ml4ca_env* env, const float* motion, const float* rate, const float* omega, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  const WaveParams& w = env->wave;
  ML4CA_REQUIRE(w.motion != nullptr, "waves are not enabled (ml4ca_env_set_waves)");
  DeviceGuard guard(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t row = (size_t)env->n * sizeof(float);
  if (motion) ML4CA_CUDA(cudaMemcpyAsync(w.motion, motion, 3 * row, cudaMemcpyDeviceToDevice, st));
  if (rate) ML4CA_CUDA(cudaMemcpyAsync(w.rate, rate, 3 * row, cudaMemcpyDeviceToDevice, st));
  if (omega) ML4CA_CUDA(cudaMemcpyAsync(w.omega, omega, row, cudaMemcpyDeviceToDevice, st));
  return ML4CA_OK;
}

int ml4ca_env_get_waves(ml4ca_env* env, float* motion, float* rate, float* omega, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  const WaveParams& w = env->wave;
  ML4CA_REQUIRE(w.motion != nullptr, "waves are not enabled (ml4ca_env_set_waves)");
  DeviceGuard guard(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t row = (size_t)env->n * sizeof(float);
  if (motion) ML4CA_CUDA(cudaMemcpyAsync(motion, w.motion, 3 * row, cudaMemcpyDeviceToDevice, st));
  if (rate) ML4CA_CUDA(cudaMemcpyAsync(rate, w.rate, 3 * row, cudaMemcpyDeviceToDevice, st));
  if (omega) ML4CA_CUDA(cudaMemcpyAsync(omega, w.omega, row, cudaMemcpyDeviceToDevice, st));
  return ML4CA_OK;
}

int ml4ca_env_set_observer(ml4ca_env* env, const ml4ca_observer_cfg* cfg, float* state, const float* omega_o, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  if (cfg == nullptr) {
    env->obsv.state = nullptr;
    env->obsv.omega = nullptr;
    return ML4CA_OK;
  }
  const int stv = validate_observer_cfg(cfg);
  if (stv != ML4CA_OK) return stv;
  ML4CA_REQUIRE(state != nullptr && omega_o != nullptr, "state [15, n] and omega_o [n] are required");
  ML4CA_REQUIRE(cfg->step_dt == env->cfg.step_dt, "the observer's step_dt must equal the env's step_dt");
  DeviceGuard guard(env->device);
  ObserverParams ob;
  ob.state = state;
  ob.omega = omega_o;
  ob.k = observer_consts(*cfg);
  attach_observer_kernel<<<(unsigned)((env->n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(env->p, env->wave, ob);
  const int rc = check_launch("attach_observer_kernel");
  if (rc == ML4CA_OK) env->obsv = ob;
  return rc;
}

int ml4ca_env_set_refmodel(ml4ca_env* env, const ml4ca_refmodel_cfg* cfg, float* state, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  if (cfg == nullptr) {
    env->refm.state = nullptr;
    return ML4CA_OK;
  }
  RefParams rf;
  const int stv = refmodel_consts(cfg, rf.k);
  if (stv != ML4CA_OK) return stv;
  ML4CA_REQUIRE(state != nullptr, "state [9, n] is required");
  ML4CA_REQUIRE(cfg->step_dt == env->cfg.step_dt, "the reference model's step_dt must equal the env's step_dt");
  DeviceGuard guard(env->device);
  rf.state = state;
  attach_refmodel_kernel<<<(unsigned)((env->n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(env->p, rf);
  const int rc = check_launch("attach_refmodel_kernel");
  if (rc == ML4CA_OK) env->refm = rf;
  return rc;
}

int ml4ca_env_set_ref(ml4ca_env* env, const float* ref, void* stream) {
  ML4CA_REQUIRE(env != nullptr && ref != nullptr, "env and ref are required");
  DeviceGuard guard(env->device);
  ML4CA_CUDA(cudaMemcpyAsync(env->p.ref, ref, 3 * (size_t)env->n * sizeof(float), cudaMemcpyDeviceToDevice,
                             static_cast<cudaStream_t>(stream)));
  return ML4CA_OK;
}

int ml4ca_env_step(ml4ca_env* env, const float* action, float* obs, float* rew, uint8_t* done, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  ML4CA_REQUIRE(action != nullptr && obs != nullptr && rew != nullptr && done != nullptr,
                "action, obs, rew and done are required");
  DeviceGuard guard(env->device);
  env->tail_valid = false;   // the tail of the returned observation now lives in the caller's obs buffer only
  return launch_step(env, 0, env->n, env->n, action, obs, rew, done, static_cast<cudaStream_t>(stream));
}

// ---- host-buffer step: chunked three-stage pipeline (H2D | kernel | D2H on three streams, two slots) -------------
int ml4ca_env_step_host(ml4ca_env* env, const float* action_host, float* obs_host, float* rew_host,
                        uint8_t* done_host, void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  ML4CA_REQUIRE(action_host != nullptr && obs_host != nullptr && rew_host != nullptr && done_host != nullptr,
                "action, obs, rew and done host buffers are required");
  DeviceGuard guard(env->device);
  int32_t act_dim = 0, obs_dim = 0;
  ml4ca_env_dims(&env->cfg, &act_dim, &obs_dim);
  HostPipe*& hp = env->pipe;
  const int64_t n = env->n;
  if (hp == nullptr) {
    hp = new (std::nothrow) HostPipe();
    ML4CA_REQUIRE(hp != nullptr, "out of host memory");
    static const int64_t chunk_pref = [] {   // tuning knob: envs per pipeline chunk
      const char* e = getenv("ML4CA_HOST_CHUNK");
      int64_t c = e ? (int64_t)atoll(e) : (int64_t)1 << 20;
      if (c < 4) c = (int64_t)1 << 20;          // 0 / negative / garbage: the loop below would never advance
      return (c + 3) / 4 * 4;                   // rows of a chunk stay 16-byte aligned
    }();
    hp->chunk = n < chunk_pref ? ((n + 3) / 4) * 4 : chunk_pref;
    const size_t per_slot = (size_t)hp->chunk * ((size_t)(act_dim + obs_dim + 1) * sizeof(float) + 1) + 64;
    ML4CA_CUDA(cudaMalloc(&hp->slab, 2 * per_slot));
    for (int s = 0; s < 2; ++s) {
      uint8_t* base = static_cast<uint8_t*>(hp->slab) + s * per_slot;
      hp->act[s] = reinterpret_cast<float*>(base);
      hp->obs[s] = hp->act[s] + (size_t)act_dim * hp->chunk;
      hp->rew[s] = hp->obs[s] + (size_t)obs_dim * hp->chunk;
      hp->done[s] = reinterpret_cast<uint8_t*>(hp->rew[s] + hp->chunk);
      ML4CA_CUDA(cudaEventCreateWithFlags(&hp->ev_in[s], cudaEventDisableTiming));
      ML4CA_CUDA(cudaEventCreateWithFlags(&hp->ev_k[s], cudaEventDisableTiming));
      ML4CA_CUDA(cudaEventCreateWithFlags(&hp->ev_out[s], cudaEventDisableTiming));
    }
    ML4CA_CUDA(cudaEventCreateWithFlags(&hp->ev_start, cudaEventDisableTiming));
    ML4CA_CUDA(cudaStreamCreateWithFlags(&hp->s_in, cudaStreamNonBlocking));
    ML4CA_CUDA(cudaStreamCreateWithFlags(&hp->s_k, cudaStreamNonBlocking));
    ML4CA_CUDA(cudaStreamCreateWithFlags(&hp->s_out, cudaStreamNonBlocking));
  }
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  ML4CA_CUDA(cudaEventRecord(hp->ev_start, user));          // everything queued on the caller's stream comes first
  ML4CA_CUDA(cudaStreamWaitEvent(hp->s_in, hp->ev_start, 0));
  ML4CA_CUDA(cudaStreamWaitEvent(hp->s_k, hp->ev_start, 0));
  env->tail_valid = false;
  const int64_t C = hp->chunk;
  const size_t hpitch = (size_t)n * sizeof(float), dpitch = (size_t)C * sizeof(float);
  int64_t k = 0;
  for (int64_t first = 0; first < n; first += C, ++k) {
    const int s = (int)(k & 1);
    const int64_t cnt = n - first < C ? n - first : C;
    if (k >= 2) ML4CA_CUDA(cudaStreamWaitEvent(hp->s_in, hp->ev_k[s], 0));      // kernel k-2 has consumed act[s]
    ML4CA_CUDA(cudaMemcpy2DAsync(hp->act[s], dpitch, action_host + first, hpitch, (size_t)cnt * sizeof(float),
                                 (size_t)act_dim, cudaMemcpyHostToDevice, hp->s_in));
    ML4CA_CUDA(cudaEventRecord(hp->ev_in[s], hp->s_in));
    ML4CA_CUDA(cudaStreamWaitEvent(hp->s_k, hp->ev_in[s], 0));
    if (k >= 2) ML4CA_CUDA(cudaStreamWaitEvent(hp->s_k, hp->ev_out[s], 0));     // copy-out k-2 has drained obs[s]
    int rc = launch_step(env, first, cnt, C, hp->act[s], hp->obs[s], hp->rew[s], hp->done[s], hp->s_k);
    if (rc != ML4CA_OK) return rc;
    ML4CA_CUDA(cudaEventRecord(hp->ev_k[s], hp->s_k));
    ML4CA_CUDA(cudaStreamWaitEvent(hp->s_out, hp->ev_k[s], 0));
    ML4CA_CUDA(cudaMemcpy2DAsync(obs_host + first, hpitch, hp->obs[s], dpitch, (size_t)cnt * sizeof(float),
                                 (size_t)obs_dim, cudaMemcpyDeviceToHost, hp->s_out));
    ML4CA_CUDA(cudaMemcpyAsync(rew_host + first, hp->rew[s], (size_t)cnt * sizeof(float), cudaMemcpyDeviceToHost,
                               hp->s_out));
    ML4CA_CUDA(cudaMemcpyAsync(done_host + first, hp->done[s], (size_t)cnt, cudaMemcpyDeviceToHost, hp->s_out));
    ML4CA_CUDA(cudaEventRecord(hp->ev_out[s], hp->s_out));
  }
  // the caller's stream resumes when the last copies have landed (the other slot finished earlier on s_out)
  ML4CA_CUDA(cudaStreamWaitEvent(user, hp->ev_out[(int)((k - 1) & 1)], 0));
  return ML4CA_OK;
}

int ml4ca_env_observe(ml4ca_env* env, float* obs, void* stream) {
  ML4CA_REQUIRE(env != nullptr && obs != nullptr, "env and obs are required");
  ML4CA_REQUIRE(!env->cfg.extended_state || env->tail_valid,
                "the previous-thrust tail of the observation is only kept by reset and ml4ca_rollout_step; after "
                "ml4ca_env_step the observation lives in the caller's obs buffer");
  DeviceGuard guard(env->device);
  observe_kernel<<<(unsigned)((env->n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      env->p, env->cfg.extended_state, obs, env->wave, env->obsv, env->refm);
  return check_launch("observe_kernel");
}

int ml4ca_env_get_state(ml4ca_env* env, float* eta, float* nu, float* prev_thrust, float* angles, int32_t* ep_len,
                        void* stream) {
  ML4CA_REQUIRE(env != nullptr, "env is NULL");
  DeviceGuard guard(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t row3 = 3 * (size_t)env->n * sizeof(float);
  if (eta) ML4CA_CUDA(cudaMemcpyAsync(eta, env->p.eta, row3, cudaMemcpyDeviceToDevice, st));
  if (nu) ML4CA_CUDA(cudaMemcpyAsync(nu, env->p.nu, row3, cudaMemcpyDeviceToDevice, st));
  if (prev_thrust) ML4CA_CUDA(cudaMemcpyAsync(prev_thrust, env->p.prev_thrust, row3, cudaMemcpyDeviceToDevice, st));
  if (angles) ML4CA_CUDA(cudaMemcpyAsync(angles, env->p.angles, row3, cudaMemcpyDeviceToDevice, st));
  if (ep_len) {
    unpack_ep_len_kernel<<<(unsigned)((env->n + 255) / 256), 256, 0, st>>>(env->n, env->p.ep_len, ep_len);
    return check_launch("unpack_ep_len_kernel");
  }
  return ML4CA_OK;
}

int ml4ca_error_frame(int64_t n, const float* eta, const float* ref, float* err, void* stream) {
  ML4CA_REQUIRE(n >= 0 && eta && ref && err, "bad arguments");
  if (n == 0) return ML4CA_OK;
  error_frame_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, eta, ref, err);
  return check_launch("error_frame_kernel");
}

int ml4ca_scale_and_clip(const ml4ca_env_cfg* cfg, int64_t n, const float* action, float* act_env, int8_t* sat,
                         void* stream) {
  int stv = validate_cfg(cfg);
  if (stv != ML4CA_OK) return stv;
  ML4CA_REQUIRE(n >= 0 && action && act_env, "bad arguments");
  if (n == 0) return ML4CA_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  switch (cfg->kind) {
    case ML4CA_ENV_FULL: scale_clip_kernel<ML4CA_ENV_FULL, false><<<blocks, 256, 0, st>>>(n, action, act_env, sat); break;
    case ML4CA_ENV_SIMPLE: scale_clip_kernel<ML4CA_ENV_SIMPLE, false><<<blocks, 256, 0, st>>>(n, action, act_env, sat); break;
    case ML4CA_ENV_LIMITED: scale_clip_kernel<ML4CA_ENV_LIMITED, false><<<blocks, 256, 0, st>>>(n, action, act_env, sat); break;
    default:
      if (cfg->cont_ang) scale_clip_kernel<ML4CA_ENV_FINAL, true><<<blocks, 256, 0, st>>>(n, action, act_env, sat);
      else scale_clip_kernel<ML4CA_ENV_FINAL, false><<<blocks, 256, 0, st>>>(n, action, act_env, sat);
  }
  return check_launch("scale_clip_kernel");
}

}  // extern "C"
