/* ml4ca_b200.h -- C ABI of libml4ca_b200.so: the B200-native ReVolt dynamic-positioning hot path.
 *
 * The reference (simensov/ml4ca) is pure Python and has no FFI layer; the seams this ABI replaces are the
 * Python call signatures listed per function below (paths relative to /root/reference).  INTEGRATION.md shows
 * the ctypes stub a reference maintainer would add at each seam.
 *
 * Conventions
 *  - every function returns 0 on success or a negative ml4ca_status; nothing throws across the ABI;
 *    ml4ca_last_error() gives the message of the last failure on the calling thread.
 *  - all data pointers are DEVICE pointers owned by the caller (e.g. PyTorch allocations) unless the
 *    parameter name ends in _host; the library owns only the opaque handles' struct-of-arrays state.
 *  - batches are struct-of-arrays, row-major [component, n]: component c of env i lives at p[c * n + i].
 *  - calls are asynchronous and ordered on `stream` (a cudaStream_t passed as void*; NULL = legacy default
 *    stream); no hidden synchronisation, no CPU fallback: without a CUDA device every compute entry fails.
 *  - one handle per device; a handle is not thread-safe, different handles are independent.
 */
#ifndef ML4CA_B200_H_
#define ML4CA_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define ML4CA_API __attribute__((visibility("default")))
#else
#define ML4CA_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  ML4CA_OK = 0,
  ML4CA_ERR_INVALID = -1, /* bad argument (the reference raises AssertionError, customEnv.py:35,228,238) */
  ML4CA_ERR_CUDA = -2,    /* CUDA runtime failure, message in ml4ca_last_error */
  ML4CA_ERR_NO_DEVICE = -3,
  ML4CA_ERR_UNSUPPORTED = -4
} ml4ca_status;

/* env kinds = the four reference env classes (customEnv.py:11,327,351,373) */
enum { ML4CA_ENV_FULL = 0, ML4CA_ENV_SIMPLE = 1, ML4CA_ENV_LIMITED = 2, ML4CA_ENV_FINAL = 3 };

/* done flags written by ml4ca_env_step */
enum { ML4CA_DONE_TERMINAL = 1, /* Revolt.is_terminal, customEnv.py:207-213 */
       ML4CA_DONE_TRUNCATED = 2 /* traj_len == max_ep_len, ppo.py:304 */ };

typedef struct ml4ca_env_cfg {
  int32_t kind;           /* ML4CA_ENV_* */
  int32_t cont_ang;       /* RevoltFinal(cont_ang=True): 7 network actions, sin/cos azimuths (customEnv.py:227-235) */
  int32_t extended_state; /* obs 9 (= 6 + previous thrust) instead of 6 (customEnv.py:201-205) */
  int32_t n_substeps;     /* simulator sub-steps of sim_dt per env step (20, customEnv.py:79-81); 0 = null simulator */
  int32_t max_ep_len;     /* 400 at 5 Hz (customEnv.py:83) */
  int32_t auto_reset;     /* 0: reference semantics (caller resets).  1: an env whose done != 0 is re-sampled inside
                             step and the returned obs is the first obs of its next episode */
  int32_t reset_acts;     /* Revolt(reset_acts=True), customEnv.py:179-188: every reset draws the previous thrust
                             as scale_and_clip(N(0, 0.1)^3) instead of [0, 0, 0] (:190); default 0 */
  int32_t hull_model;     /* stand-in hull parameter set (DECLARED, ml4ca_constants.h): 0 = round-1 constants, 1 = the
                             constants fitted to the reference's recorded box tests (tools/sysid_hull.py) */
  float ss_bounds[6];     /* termination bounds real_ss_bounds (customEnv.py:26,337,361,386) */
  float sim_dt;           /* 0.01 s */
  float step_dt;          /* dt used by the action-derivative penalty = 0.01 * 20 (customEnv.py:81,311,317) */
  float reset_fraction;   /* fraction used by auto_reset (0.8, ppo.py:286,320) */
  float actuator_lag_s;   /* > 0: the thruster wrench follows its command through a first-order lag of this time constant,
                             advanced every simulator sub-step (three more state rows).
                             0 (default): commanded thrust / azimuth act instantly */
  uint64_t seed;          /* Philox key */
  int64_t env_id_offset;  /* global id of local env 0: RNG streams do not depend on how envs shard over GPUs */
} ml4ca_env_cfg;

typedef struct ml4ca_env ml4ca_env;

/* Reference defaults for one env class.  Replaces Revolt.__init__ / RevoltSimple / RevoltLimited / RevoltFinal
 * (src/rl/windows_workspace/specific/customEnv.py:22-90,331-349,355-371,377-399). */
ML4CA_API int ml4ca_env_cfg_default(int32_t kind, int32_t cont_ang, int32_t extended_state, ml4ca_env_cfg* out);
/* dims implied by a cfg: network action dim (3/5/6/7) and obs dim (6/9) */
ML4CA_API int ml4ca_env_dims(const ml4ca_env_cfg* cfg, int32_t* act_dim, int32_t* obs_dim);

ML4CA_API int ml4ca_env_create(const ml4ca_env_cfg* cfg, int64_t n_env, int32_t device, ml4ca_env** out);
ML4CA_API int ml4ca_env_destroy(ml4ca_env* env);

/* Revolt.reset(fraction=...) in training mode (customEnv.py:135-194; samplers simtools.py:109-124).
 * mask [n] (nullable = all): envs to reset.  obs [obs_dim, n]: written for the reset envs only. */
ML4CA_API int ml4ca_env_reset(ml4ca_env* env, const uint8_t* mask, float fraction, float* obs, void* stream);
/* Revolt.reset(**init) with explicit 'Hull.PosNED/PosAttitude/VelocityNu' (customEnv.py:141-161):
 * eta [3, n] = N, E, yaw; nu [3, n] = u, v, r. */
ML4CA_API int ml4ca_env_reset_to(ml4ca_env* env, const uint8_t* mask, const float* eta, const float* nu, float* obs,
                       void* stream);
/* Side buffer for the value bootstrap at the episode-length cut (ppo.py:303-311: `last_val = 0 if d else v(o)` on the
 * observation o2 that env.step returned).  With auto_reset the in-kernel restart replaces that observation in the step's
 * output; cut_obs [obs_dim, n] (caller-owned device memory, NULL = off) receives it instead, for the envs whose flag byte
 * is exactly ML4CA_DONE_TRUNCATED; other columns are left untouched. */
ML4CA_API int ml4ca_env_set_cut_obs(ml4ca_env* env, float* cut_obs);
/* The `fraction` every later in-kernel restart samples with (curriculum learning, ppo.py:286,319-322: the reference passes
 * it to each env.reset).  Launch parameter: CUDA graphs captured earlier keep the value they were captured with. */
ML4CA_API int ml4ca_env_set_reset_fraction(ml4ca_env* env, float fraction);
/* ErrorFrame.update(ref=new_ref) (errorFrame.py:34-38; customEnv.py:131,155-156): ref [3, n]. */
ML4CA_API int ml4ca_env_set_ref(ml4ca_env* env, const float* ref, void* stream);
/* Revolt.step(action) (customEnv.py:92-133): action [act_dim, n] -> obs [obs_dim, n], rew [n], done [n] flags. */
ML4CA_API int ml4ca_env_step(ml4ca_env* env, const float* action, float* obs, float* rew, uint8_t* done, void* stream);
/* The same step for callers whose buffers live in HOST memory (the reference's callers hold NumPy arrays:
 * ppo.py:291-293 feeds `a[0]` to env.step and reads o, r, d back).  action_host [act_dim, n], obs_host [obs_dim, n],
 * rew_host [n], done_host [n]; page-locked buffers give full overlap.  The batch is cut into chunks that run through
 * a three-stage pipeline on library-owned streams (host->device copy | kernel | device->host copy), so that both
 * PCIe directions and the SMs are busy at once.  Ordered after the work already queued on `stream`; `stream`
 * resumes when the last result bytes have landed (synchronise it before reading the host buffers). */
ML4CA_API int ml4ca_env_step_host(ml4ca_env* env, const float* action_host, float* obs_host, float* rew_host,
                                  uint8_t* done_host, void* stream);
/* Revolt.state() / state_extended() (customEnv.py:196-205) of the current state: obs [obs_dim, n].  With the extended
 * state this needs the previous-thrust tail, which the library keeps after reset only. */
ML4CA_API int ml4ca_env_observe(ml4ca_env* env, float* obs, void* stream);
/* Copies of the SoA state (any pointer may be NULL): eta [3,n], nu [3,n], prev_thrust [3,n] (env order bow, port,
 * star), angles [3,n] (current_angles, customEnv.py:71), ep_len [n].  Also EF.get_NED_pos (errorFrame.py:19). */
ML4CA_API int ml4ca_env_get_state(ml4ca_env* env, float* eta, float* nu, float* prev_thrust, float* angles, int32_t* ep_len,
                        void* stream);
ML4CA_API int64_t ml4ca_env_size(const ml4ca_env* env);

/* Environmental disturbance (DECLARED model, DESIGN.md section 4; the reference's Cybersea simulator sets its environment
 * through DigiTwin.val, digitwin.py:213-217).  Ocean current: constant in the NED frame over an episode,
 * v_c = V [cos beta, sin beta] with V ~ U(current_speed_min, current_speed_max) and beta ~ U(current_dir_min,
 * current_dir_max) drawn at every reset (explicit or in-kernel); beta is the direction the water flows towards (0 = north,
 * pi/2 = east).  The hull equations act on the velocity relative to the water; the observed nu stays the velocity over
 * ground.  Bias force: b = [X_N, Y_E, N_psi] in the NED frame, a first-order Gauss-Markov process
 * b <- a b + bias_std sqrt(1 - a^2) w per env step, a = exp(-step_dt / bias_time_s), drawn as b = bias_std w0 at every reset;
 * bias_time_s = 0 keeps b constant over the episode.  Holding station against a beam current of 0.3 m/s takes the full sway
 * thrust of either hull model: 0 to 0.2 m/s is the useful range. */
typedef struct ml4ca_disturbance_cfg {
  float current_speed_min, current_speed_max; /* m/s, 0 <= min <= max */
  float current_dir_min, current_dir_max;     /* rad, min <= max */
  float bias_std[3];                          /* N, N, Nm, >= 0: stationary standard deviation of b */
  float bias_time_s;                          /* >= 0: time constant of b; 0 = constant over the episode */
} ml4ca_disturbance_cfg;

/* Enable (cfg != NULL) or switch off (cfg = NULL) the disturbance.  Enabling draws the current and the bias of every env
 * from the new ranges on `stream`; every later reset draws them again.  Launch parameter: CUDA graphs captured earlier
 * keep the values they were captured with.  Bad ranges: ML4CA_ERR_INVALID. */
ML4CA_API int ml4ca_env_set_disturbance(ml4ca_env* env, const ml4ca_disturbance_cfg* cfg, void* stream);
/* Overwrite the disturbance state: current [2, n] (NED, m/s) and bias [3, n] (N, N, Nm), either nullable.  The values hold
 * until that env's next reset.  Needs an enabled disturbance. */
ML4CA_API int ml4ca_env_set_disturbance_state(ml4ca_env* env, const float* current, const float* bias, void* stream);
/* Copies of the disturbance state: current [2, n], bias [3, n], either nullable.  Needs an enabled disturbance. */
ML4CA_API int ml4ca_env_get_disturbance(ml4ca_env* env, float* current, float* bias, void* stream);

/* First-order wave-frequency motion (DECLARED model, DESIGN.md section 4; set at the same DigiTwin.val seam).  Per env
 * and DOF d (surge, sway, yaw; body frame) a linear oscillator driven by white noise,
 * x'' + 2 lambda w0 x' + w0^2 x = sigma_d sqrt(4 lambda w0^3) w(t), with stationary std sigma_d of x and w0 sigma_d of x'.
 * w0 ~ U(omega_min, omega_max) is drawn at every reset (explicit or in-kernel) together with a stationary state; the state
 * then takes one exact step per env step (also with n_substeps = 0).  The motion never moves the hull: eta and nu stay
 * the low-frequency state.  The observation, the reward and the termination of every step and reset, cut_obs and
 * ml4ca_env_observe see the measured values N + cos(psi) x_s - sin(psi) x_w, E + sin(psi) x_s + cos(psi) x_w,
 * psi + x_psi and nu + x'. */
typedef struct ml4ca_wave_cfg {
  float sigma[3];             /* m, m, rad, >= 0: stationary std of the WF motion in surge, sway, yaw (body frame) */
  float omega_min, omega_max; /* rad/s, 0 < min <= max, max * step_dt < pi: peak frequency, drawn per episode */
  float damping;              /* 0 < lambda < 1 */
} ml4ca_wave_cfg;
/* cfg = NULL switches waves off (rows stay allocated).  Enabling draws every env's state on `stream`.  Launch
 * parameter, like the restart fraction and the disturbance: CUDA graphs captured earlier keep theirs.  Bad values:
 * ML4CA_ERR_INVALID. */
ML4CA_API int ml4ca_env_set_waves(ml4ca_env* env, const ml4ca_wave_cfg* cfg, void* stream);
/* motion [3, n], rate [3, n] (body frame), omega [n]; any may be NULL; needs enabled waves.  Set values hold until that
 * env's next reset. */
ML4CA_API int ml4ca_env_set_wave_state(ml4ca_env* env, const float* motion, const float* rate, const float* omega,
                                       void* stream);
/* Copies of the wave state: motion [3, n], rate [3, n], omega [n]; any may be NULL; needs enabled waves. */
ML4CA_API int ml4ca_env_get_waves(ml4ca_env* env, float* motion, float* rate, float* omega, void* stream);

/* Stateless pieces of the wrapper, exposed for callers that own their own state (and for parity tests):
 * ErrorFrame.transform (errorFrame.py:25-32): eta, ref [3, n] -> err [3, n] body-frame error. */
ML4CA_API int ml4ca_error_frame(int64_t n, const float* eta, const float* ref, float* err, void* stream);
/* handle_continuous_angles / wrap_stern_angles + scale_and_clip (customEnv.py:215-244; ROS twin
 * src/rl/ROS/rl_allocator/src/rl_allocator.py:222-226,275-283): action [act_dim, n] -> act_env [k, n]
 * (k = 3/5/6 real commands) and sat [k, n] (-1/0/+1 = clipped low / inside / clipped high). */
ML4CA_API int ml4ca_scale_and_clip(const ml4ca_env_cfg* cfg, int64_t n, const float* action, float* act_env, int8_t* sat,
                         void* stream);

/* Pseudoinverse allocator + DP PID controller.  ABSENT from the reference (DNV GL's dp_controller package, only
 * referenced at qp_allocator.py:6,83 and SupervisedTau.py:37); equations are this build's own, see DESIGN.md.
 * eta, nu, ref [3, n]; integ [3, n] in/out integral state; tau [3, n] (nullable) saturated PID wrench;
 * n_pct [3, n] thrust in percent, allocator order port, star, bow; alpha [2, n] stern azimuths. */
ML4CA_API int ml4ca_pinv_pid(int64_t n, const float* eta, const float* nu, const float* ref, float* integ, float* tau,
                   float* n_pct, float* alpha, void* stream);
/* Allocation only: tau [3, n] -> n_pct [3, n], alpha [2, n]. */
ML4CA_API int ml4ca_pinv_allocate(int64_t n, const float* tau, float* n_pct, float* alpha, void* stream);

/* Passive nonlinear DP observer (Fossen & Strand 1999; Fossen 2011 section 11.4.1), the state estimator between the sensors
 * and the controller of a DP stack.  ABSENT from the reference like the PID (dp_controller); declared model, DESIGN.md
 * section 4.  Per env it removes the wave-frequency part of the measured pose y [3, n] (N, E, psi), and estimates the
 * low-frequency pose, the low-frequency body velocity and the slowly varying environmental force (NED, N, N, Nm: the frame
 * and units of the env's bias).  Inputs of a step: y after the env step, and the thrust [3, n] (%) and azimuths
 * angles [3, n] (rad) that step applied, env order bow, port, star (ml4ca_env_get_state's prev_thrust and angles).
 * state [15, n] (caller-owned) rows: xi1^[3], xi2^[3] (wave states; xi2^ is the WF pose estimate), eta^[3], nu^[3], b^[3].
 * omega_o [n]: the observer's wave peak frequency per env (a fixed tuning or the env's wave_omega); values outside
 * [0.1, 10] rad/s, NaN included, are clamped into it (NaN -> 0.1).  The kinetic model is the declared hull hull_model
 * without actuator lag; the rotation uses the measured heading, held over the step. */
typedef struct ml4ca_observer_cfg {
  int32_t hull_model;  /* 0 / 1: the declared hull of the kinetic model */
  float step_dt;       /* s, > 0: n_sub = max(1, round(step_dt / 0.01)) sub-steps of step_dt / n_sub */
  float notch_damping; /* zeta_n > wave_damping */
  float wave_damping;  /* lambda, 0 < lambda < 1 */
  float cutoff_ratio;  /* omega_c / omega_o > 1 */
  float bias_time_s;   /* >= 0, 0 = infinity */
  float k3[3], k4[3];  /* >= 0: bias and velocity injection gains per DOF */
} ml4ca_observer_cfg;
/* The declared defaults (ml4ca_constants.h ML4CA_OBS_*) for hull_model 0 or 1.  Host-only. */
ML4CA_API int ml4ca_observer_cfg_default(int32_t hull_model, ml4ca_observer_cfg* cfg);
/* eta^ = y, xi^ = nu^ = b^ = 0 for every env whose mask byte is non-zero (mask = NULL: all). */
ML4CA_API int ml4ca_observer_reset(int64_t n, const float* y, const uint8_t* mask, float* state, void* stream);
/* One env step.  restart [n] (nullable): an env whose byte is non-zero is re-initialised from this y (as by
 * ml4ca_observer_reset) instead of stepped: pass the done-flag byte of an auto_reset env.  Bad configurations or
 * arguments: ML4CA_ERR_INVALID.  n = 0: no launch. */
ML4CA_API int ml4ca_observer_step(const ml4ca_observer_cfg* cfg, int64_t n, const float* y, const float* thrust,
                                  const float* angles, const float* omega_o, const uint8_t* restart, float* state,
                                  void* stream);
/* DP observer in the loop: attach (cfg != NULL) or detach (cfg = NULL) an observer that every env step runs inside the
 * step kernel.  state [15, n] and omega_o [n] are caller-owned, laid out as for ml4ca_observer_step, and must outlive the
 * attachment.  cfg->step_dt must equal the env's step_dt; the hull model may differ from the env's (a model-mismatch
 * experiment).  Attaching re-initialises every env's column from its current measured pose on `stream`.
 * While attached, each step advances the column once with y = the measured pose after the step (LF pose plus waves) and
 * the thrust and azimuths the step applied, and the observation rows 0-5 are error_frame(eta^, ref) and nu^.  Rows 6-8,
 * the reward, the flags and the env state are unchanged: the observer changes only what the agent sees.  cut_obs holds the
 * estimate-based observation of the cut step (after the update, before the restart).  An in-kernel restart, a reset or
 * reset_to re-initialises the env's column from the new measured pose (eta^ = y, the rest 0; the returned nu^ is 0), and
 * ml4ca_env_observe returns rows 0-5 from the current eta^ and nu^.  Cost: 124 B more per env-step (read 60 + 4, write
 * 60), e.g. 229 -> 353 B for RevoltFinal (extended, continuous angles) in waves.  Launch parameter: CUDA graphs
 * captured earlier keep theirs.  Bad configurations, NULL state or omega_o, a step_dt mismatch: ML4CA_ERR_INVALID. */
ML4CA_API int ml4ca_env_set_observer(ml4ca_env* env, const ml4ca_observer_cfg* cfg, float* state, const float* omega_o,
                                     void* stream);

/* DP reference model (guidance; Fossen 2011 section 12.1): per env and per DOF (N, E, psi; NED) a third-order filter with
 * saturating elements that turns a set-point r [3, n] into a smooth desired pose eta_d, velocity v_d (NED rates) and
 * acceleration a_d for the controller.  Declared model, DESIGN.md section 4 "DP reference model":
 *   eta_d / r = w^3 / ((s + w)(s^2 + 2 zeta w s + w^2)),  jerk = w^3 e - (2 zeta + 1) w a_d - (2 zeta + 1) w^2 v_d,
 *   e = r - eta_d (heading: e wrapped to [-pi, pi), eta_d,psi itself is not wrapped).
 * r is held over the env step; n_sub = max(1, round(step_dt / 0.01)) semi-implicit Euler sub-steps of h = step_dt / n_sub:
 *   a_d <- clamp(a_d + h jerk, +-a_max),  v_d <- clamp(v_d + h a_d, +-v_max),  eta_d <- eta_d + h v_d.
 * state [9, n] (caller-owned) rows: eta_d[3], v_d[3], a_d[3].
 * Validation: every value finite and > 0, and per DOF the linear sub-step map stable: with q = h omega, c = 2 zeta + 1 its
 * characteristic polynomial z^3 + a2 z^2 + a1 z + a0 (a2 = q^3 + c q^2 + c q - 3, a1 = 3 - 2 c q - c q^2, a0 = c q - 1)
 * must meet the Jury conditions p(1) > 0, p(-1) < 0, |a0| < 1, |a0^2 - 1| > |a0 a2 - a1|.  Otherwise ML4CA_ERR_INVALID. */
typedef struct ml4ca_refmodel_cfg {
  float step_dt;  /* s, > 0 */
  float zeta[3];  /* relative damping of the mass-spring-damper part, per DOF */
  float omega[3]; /* rad/s, natural frequency (and low-pass corner) per DOF */
  float v_max[3]; /* m/s, m/s, rad/s */
  float a_max[3]; /* m/s^2, m/s^2, rad/s^2 */
} ml4ca_refmodel_cfg;
/* The declared defaults (ml4ca_constants.h ML4CA_REF_*) at step_dt = 0.2 s.  Host-only. */
ML4CA_API int ml4ca_refmodel_cfg_default(ml4ca_refmodel_cfg* cfg);
/* eta_d = eta0 [3, n], v_d = a_d = 0.  n = 0: no launch. */
ML4CA_API int ml4ca_refmodel_reset(int64_t n, const float* eta0, float* state, void* stream);
/* One env step of every env's filter toward its set-point [3, n].  Bad configurations or arguments: ML4CA_ERR_INVALID.
 * n = 0: no launch. */
ML4CA_API int ml4ca_refmodel_step(const ml4ca_refmodel_cfg* cfg, int64_t n, const float* setpoint, float* state,
                                  void* stream);
/* ml4ca_pinv_pid with velocity feed-forward: v_d [3, n] (NED rates, e.g. rows 3-5 of a reference model's state) turns the
 * D-term into Kd (nu - R(psi)^T v_d), psi = eta[2].  Other arguments as ml4ca_pinv_pid; v_d is required. */
ML4CA_API int ml4ca_pinv_pid_ff(int64_t n, const float* eta, const float* nu, const float* ref, const float* v_d,
                                float* integ, float* tau, float* n_pct, float* alpha, void* stream);
/* DP reference model in the loop: attach (cfg != NULL) or detach (cfg = NULL) a reference model that every env step runs
 * inside the step kernel.  state [9, n] is caller-owned, laid out as for ml4ca_refmodel_step, and must outlive the
 * attachment.  cfg is validated as by ml4ca_refmodel_step (Jury test included) and cfg->step_dt must equal the env's
 * step_dt.  Attaching re-initialises every env's column from its current LF pose (eta_d = eta, v_d = a_d = 0) on `stream`.
 * While attached, the env's set-point rows (ml4ca_env_set_ref) hold the operator's command s.  Each step first advances
 * the env's column once on s (eta_d(t) -> eta_d(t+1), the arithmetic of ml4ca_refmodel_step), and then forms everything
 * it forms against the set-point against eta_d(t+1) instead: observation rows 0-2 (and an attached observer's error
 * frame), the reward and the termination.  Rows 3-8 are unchanged; the reward's velocity penalty still acts on nu.  So a
 * step equals, bit for bit, ml4ca_refmodel_step on s, ml4ca_env_set_ref(eta_d) and a step without the model.  cut_obs is
 * formed after this step's advance and before the restart.  An in-kernel restart, a reset or reset_to starts the env's
 * column again at the new episode's LF pose (not the measured one), and ml4ca_env_observe forms rows 0-2 against the
 * current eta_d.  Cost: 72 B more per env-step (read 36, write 36), e.g. 177 -> 249 B for RevoltFinal (extended,
 * continuous angles).  Launch parameter: CUDA graphs captured earlier keep theirs.  Bad configurations, a NULL state, a
 * step_dt mismatch: ML4CA_ERR_INVALID. */
ML4CA_API int ml4ca_env_set_refmodel(ml4ca_env* env, const ml4ca_refmodel_cfg* cfg, float* state, void* stream);

/* QPTA.solve_QP (src/qp/ROS/qp_allocator/src/qp_allocator.py:108-234): tau [3, n] desired wrench, prev [5, n]
 * previous thruster state [f_port, f_star, f_bow, a_port, a_star] -> x [8, n] = [f(3), a(2), s(3)] after the
 * |x| < 0.01 clean-up (:232), status [n]: bit 0 = success (the reference's second return value; on failure the
 * caller holds the previous state, :267-269), bits 1..16 = active set at x (bits 1-5 z_i at its lower effective
 * bound, 6-10 upper, 11-13 s_i = -1, 14-16 s_i = +1), bits 17..20 = SLSQP exit mode (0 success, 4 incompatible
 * constraints, 8 positive directional derivative, 9 iteration limit), bits 24..31 = major iterations.  The solver
 * follows SLSQP's own path (csrc/qp_slsqp.cuh), in float64: same local minimum, same stopping iteration, same flag as the
 * reference.  Never fails on infeasible demands: it reports success = 0, like the reference. */
ML4CA_API int ml4ca_qp_solve(int64_t n, const float* tau, const float* prev, float* x, uint32_t* status, void* stream);
/* The objective switches of solve_QP(tau_d, weight_matrix, reduce_fuel, reduce_flickering, reduce_angular) (:108,116-150).
 * weights = diagonal of Q over obj = [s(3), fuel term (3), |a - a_prev| (2), |f - f_prev| (3)]; a term that is switched
 * off (reduce_angular / reduce_flickering = False) has weight 0.  Reference default (:138-148): 1,1,1, 1,1,1, .25,.25,
 * .25,.25,.25.  reduce_fuel = 0 replaces |f|^1.5 by f (:128-131).  raw = 1 skips the |x| < 0.01 clean-up (diagnostics). */
typedef struct ml4ca_qp_options {
  float weights[11];
  int32_t reduce_fuel;
  int32_t raw;
} ml4ca_qp_options;
ML4CA_API int ml4ca_qp_options_default(ml4ca_qp_options* opt);
ML4CA_API int ml4ca_qp_solve_ex(int64_t n, const float* tau, const float* prev, const ml4ca_qp_options* opt /* NULL = default */,
                                float* x, uint32_t* status, void* stream);
/* QPTA.tau_controller_callback_func (:247-320): solve + post-processing + state update.  prev [5, n] is updated
 * in place to [F, mapToPi(alpha)] (held where the solve failed); out [7, n] = thrust percent n_port, n_star, n_bow
 * (n = sign(F/K) sqrt(|F/K|), :284-288), azimuths a_port, a_star, a_bow in rad mapped to [-pi, pi) (:276-277), bow
 * throttle clip(2.5 n_bow, +-100) (:307, SIMULATION = False).  status as above (nullable). */
ML4CA_API int ml4ca_qp_allocate(int64_t n, const float* tau, float* prev, float* out, uint32_t* status, void* stream);

/* ---- PPO actor/critic MLP (spinup/algos/tf1/ppo/core.py:29-33,42-46,80-107 of src/rl/windows_workspace) ---------
 * Supported networks: hidden 64x64 (BASELINE config), 64x64x64 and 80x80x80 (the shipped checkpoints); obs_dim <= 15,
 * act_dim <= 7.  Parameters are one flat fp32 vector in the reference's variable order:
 *   pi/dense/kernel [obs,H], pi/dense/bias [H], pi/dense_1/..., pi/dense_k/kernel [H,act], bias [act], pi/log_std [act],
 *   v/dense/kernel [obs,H], ..., v/dense_k/kernel [H,1], bias [1]            (kernels row-major [in, out]). */
typedef struct ml4ca_policy_cfg {
  int32_t obs_dim, act_dim;
  int32_t hidden, n_hidden;
  int32_t activation; /* 0 tanh (core.py:94 default), 1 leaky_relu alpha 0.2 (train.py:24,31; every shipped model) */
  int32_t reserved;
} ml4ca_policy_cfg;
typedef struct ml4ca_policy ml4ca_policy;

ML4CA_API int64_t ml4ca_policy_num_params(const ml4ca_policy_cfg* cfg);
/* params_host: ml4ca_policy_num_params floats in HOST memory (NULL = zeros).  The library keeps an fp32 master copy
 * on the device and the fp16 tensor-core operand image derived from it. */
ML4CA_API int ml4ca_policy_create(const ml4ca_policy_cfg* cfg, const float* params_host, int32_t device, ml4ca_policy** out);
ML4CA_API int ml4ca_policy_destroy(ml4ca_policy* p);
/* device pointer of the fp32 master parameters (an optimizer updates them in place) ... */
ML4CA_API float* ml4ca_policy_params(ml4ca_policy* p);
/* the cfg a policy was created with, and its device */
ML4CA_API int ml4ca_policy_describe(const ml4ca_policy* p, ml4ca_policy_cfg* cfg, int32_t* device);
/* ... and re-derives the operand image afterwards */
ML4CA_API int ml4ca_policy_refresh(ml4ca_policy* p, void* stream);
/* get_action_ops = [pi, v, logp_pi] of ppo.py:221,291: obs [obs_dim, n] -> act [act_dim, n] = mu + eps * exp(log_std)
 * (eps ~ N(0,1) from Philox keyed by (seed, env_id_offset + i, step); deterministic != 0: act = mu, the evaluation
 * action pi/dense_k/BiasAdd of test_policy.py:90), val [n], logp [n], mu [act_dim, n] (nullable). */
ML4CA_API int ml4ca_policy_forward(ml4ca_policy* p, int64_t n, const float* obs, uint64_t seed, uint32_t step,
                                   int32_t deterministic, int64_t env_id_offset, float* act, float* val, float* logp,
                                   float* mu, void* stream);

/* CUDA-graph support for launch-bound rollouts (no reference counterpart: the reference steps one env per sess.run).  With a
 * device-resident counter set, every later ml4ca_policy_forward uses step + *step_dev as the Philox
 * step: a captured graph of T rollout steps (step arguments 0 .. T-1) is replayed epoch after epoch with fresh noise by
 * writing the epoch's first step number into the counter.  NULL restores the plain step argument. */
ML4CA_API int ml4ca_policy_set_step_counter(ml4ca_policy* p, const uint32_t* step_dev);
/* TrajectoryBuffer.finish_path for every environment (ppo.py:65-91; core.discount_cumsum core.py:48-63):
 * rew [T, n], val [T + 1, n] (row T = bootstrap values at the buffer end, ppo.py:311), done [T, n] flag bytes
 * (nullable) -> adv [T, n], ret [T, n].  boot [ceil(T / boot_window), n] (nullable): `last_val = v(o)` of ppo.py:311 at
 * an episode-length cut inside the buffer, i.e. V of the observation the env returned AT the cut (ml4ca_env_set_cut_obs);
 * a cut at step t reads row t / boot_window.  Two cuts of one env are >= max_ep_len steps apart, so boot_window =
 * max_ep_len keeps one row per window; boot_window = 1 is the plain [T, n] layout.  boot = NULL: V(s_t) stands in. */
ML4CA_API int ml4ca_gae(int64_t n, int32_t T, const float* rew, const float* val, const uint8_t* done, const float* boot,
                        int32_t boot_window, float gamma, float lam, float* adv, float* ret, void* stream);
/* mpi_statistics_scalar (mpi_tools.py:71-93), local part: out3 (device, 3 doubles) = [sum, sum of squares, count]. */
ML4CA_API int ml4ca_stats(int64_t m, const float* x, double* out3, void* stream);
/* ... with_min_and_max=True: out5 (device, 5 doubles) = [sum, sum of squares, count, min, max] (min / max = +-1e300 if empty). */
ML4CA_API int ml4ca_stats5(int64_t m, const float* x, double* out5, void* stream);
/* The logger's EpRet / EpLen (ppo.py:296-297,317-318; logx.EpochLogger) from the [T, n] reward and done-flag records:
 * run_ret [n], run_len [n] carry the episode in progress across epochs (in/out); ret5 / len5 as in ml4ca_stats5 over the
 * episodes that ended inside the buffer. */
ML4CA_API int ml4ca_episode_stats(int64_t n, int32_t T, const float* rew, const uint8_t* done, float* run_ret,
                                  int32_t* run_len, double* ret5, double* len5, void* stream);
/* advantage normalisation x <- (x - mean) / (std + 1e-8) (ppo.py:103). */
ML4CA_API int ml4ca_normalize(int64_t m, float* x, float mean, float std, void* stream);

/* ---- deployment-side adapters (src/rl/ROS/rl_allocator/src/rl_allocator.py, utils.py, errorFrame.py) -----------------
 * State vector of the ROS node (rl_allocator.py:165-206,215-217,252-273; ROS-twin ErrorFrame errorFrame.py:52-58, which
 * wraps radians to [-pi, pi)): eta [3, n] NED pose (yaw in rad), nu [3, n], ref [3, n], prev_u [6, n] = previous action in
 * ROS order [n_port, n_star, n_bow, a_port, a_star, a_bow] -> state [9, n] = [surge, sway, yaw error, u, v, r,
 * n_bow/100, n_port/100, n_star/100].  integ [3, n] + t_inside [n] (both nullable together) = the optional body-frame
 * integrator and the seconds spent inside its activation box (the node compares wall-clock time; h = callback period). */
ML4CA_API int ml4ca_ros_state(int64_t n, const float* eta, const float* nu, const float* ref, const float* prev_u,
                              float* integ, float* t_inside, float h, float* state, void* stream);
/* RLTA.get_action after the actor (rl_allocator.py:222-250,275-283) and create_publishable_messages (utils.py:88-115):
 * network action [act_dim, n] of env class `kind` -> u [6, n] in ROS order with the class defaults filled in, and
 * msg [7, n] (nullable) = [pod_angle.port deg, pod_angle.star deg, port_effort, star_effort, throttle_bow,
 * position_bow, lin_act_bow]; simulation = 0 is the shipped setting (bow throttle x 2.5 clipped, position 45). */
ML4CA_API int ml4ca_ros_action(int32_t kind, int32_t cont_ang, int32_t simulation, int64_t n, const float* action,
                               float* u, float* msg, void* stream);

/* Evaluation metrics of the thesis' comparison (results/all_plots/common.py:60-74, box_test/plot_pos.py:174,
 * box_test/plot_act.py:128-135,184-207,320-391) for n recorded runs of T samples at period dt: eta [T, 3, n] NED pose
 * (yaw rad), ref [3, n], thrust [T, 3, n] (bow, port, star in %), angles [T, 2, n] (port, star in rad) ->
 * out [3, n] = IAE (pose error scaled by [5 m, 5 m, 25 deg], trapezoidal), W* (propeller energy, J), IADC. */
ML4CA_API int ml4ca_eval_metrics(int64_t n, int32_t T, float dt, const float* eta, const float* ref, const float* thrust,
                                 const float* angles, float* out, void* stream);

/* Allocator output -> network-order env action, the inverse of the env's action map (customEnv.py:47-53,104-122), so
 * that the QP / pseudoinverse allocators can drive the same env as the RL policy (the thesis' three-way comparison):
 * n_pct [3, n] percent thrust port, star, bow; alpha [2, n] stern azimuths (rad) -> action [7, n] = thrusts / 100 and
 * (sin, cos) pairs (cont_ang) or action [5, n] with azimuths / ang_bound. */
ML4CA_API int ml4ca_alloc_to_action(int64_t n, int32_t cont_ang, float ang_bound, const float* n_pct, const float* alpha,
                                    float* action, void* stream);

/* ---- PPO update (ppo.py:234-250,260-280; mpi_tf.py:45-80) --------------------------------------------------------------
 * Gradient of ONE loss over a whole trajectory buffer: net 0 = pi_loss = -mean(min(ratio adv, clip(ratio) adv)) w.r.t. the
 * pi variables and log_std, net 1 = v_loss = mean((ret - v)^2) w.r.t. the v variables.  obs [T, obs_dim, n],
 * act [T, act_dim, n], adv / ret / logp_old [T, n] (the layout ml4ca_rollout_step records).  SUM convention: grad
 * (flat, parameter order, overwritten: the other net's block is zero) and stats hold sums over the LOCAL samples; the
 * caller all-reduces them over ranks and divides by the global sample count -- Allreduce(SUM) / num_procs of
 * mpi_tf.py:59-62 with equal shards.  stats (8 doubles, device): [0] sum min(ratio adv, min_adv) (= -N pi_loss),
 * [1] sum (ret - v)^2, [2] sum 0.5 (logp_old - logp)^2 (approx_kl), [3] sum -logp (approx_ent), [4] clipped count,
 * [5] sample count.  Networks: every one ml4ca_policy_create accepts -- hidden 64 x 64 (the BASELINE training config) and the
 * reference's own 80 x 80 x 80 (train.py:30-32) and 64 x 64 x 64 -- on the tcgen05 kernel, or with ml4ca_ppo_use_fp32(1) on
 * the register-tiled fp32 one (64 x 64, obs_dim <= 12) or the generic fp32 kernel (csrc/ppo_update_generic.cu: the others). */
ML4CA_API int ml4ca_ppo_grad(ml4ca_policy* p, int32_t net, int64_t n, int32_t T, const float* obs, const float* act,
                             const float* adv, const float* ret, const float* logp_old, float clip_ratio, float* grad,
                             double* stats, void* stream);
/* ---- the whole update() of ppo.py:260-280 as ONE CUDA graph ------------------------------------------------------------------
 * The early stop of the policy iterations (ppo.py:268-271: `if kl > 1.5 * target_kl: break`, after the step of that
 * iteration has been applied) needs no host round trip when the flag lives on the device: every pass of iteration i is
 * skipped when ctl->stop != 0 && ctl->stop_iter < i.  ctl is caller-owned DEVICE memory. */
typedef struct ml4ca_ppo_ctl {
  int32_t stop;        /* set by ml4ca_adam_step_dev when the rank-summed approx-KL exceeds the limit */
  int32_t stop_iter;   /* the iteration whose step was the last one applied */
  int32_t t_pi, t_v;   /* Adam step counts of the two optimizers (bias correction), advanced by ml4ca_ppo_ctl_end */
  float first[8];      /* statistics sums of iteration 0: [0..4] of the pi pass, [5] sum (ret - v)^2 of the v pass */
} ml4ca_ppo_ctl;
/* stop = 0, stop_iter = INT_MAX (start of an update; t_pi / t_v are kept). */
ML4CA_API int ml4ca_ppo_ctl_begin(ml4ca_ppo_ctl* ctl, void* stream);
/* t_pi += iterations actually applied, t_v += v_iters; stop_iter = pi_iters - 1 if the loop ran to its end. */
ML4CA_API int ml4ca_ppo_ctl_end(ml4ca_ppo_ctl* ctl, int32_t pi_iters, int32_t v_iters, void* stream);
/* ml4ca_ppo_grad that does nothing when ctl says the loop has stopped before `iter` (ctl = NULL: never skips). */
ML4CA_API int ml4ca_ppo_grad_ex(ml4ca_policy* p, int32_t net, int64_t n, int32_t T, const float* obs, const float* act,
                                const float* adv, const float* ret, const float* logp_old, float clip_ratio, float* grad,
                                double* stats, const ml4ca_ppo_ctl* ctl, int32_t iter, void* stream);
/* ml4ca_adam_step with everything the host loop decided moved to the device: the step count is ctl->t_pi (net 0) or
 * ctl->t_v (net 1) + iter + 1; skipped like ml4ca_ppo_grad_ex; stats_tail (device, 5 floats: the rank-summed statistics of
 * this iteration's pass) feeds ctl->first at iter 0 and, for net 0 with kl_limit > 0, the stop test
 * stats_tail[2] / count > kl_limit (count = global sample count; grad_scale = 1 / count). */
ML4CA_API int ml4ca_adam_step_dev(int64_t m, float* params, const float* grad, float* m1, float* m2, float lr, float beta1,
                                  float beta2, float eps, float grad_scale, int32_t net, int32_t iter, const float* stats_tail,
                                  float count, float kl_limit, ml4ca_ppo_ctl* ctl, void* stream);
/* ---- Gradient exchange over NVLink peer memory, fused with the Adam step (ranks = GPUs of one node) --------------------------
 * Replaces MpiAdamOptimizer.compute_gradients / apply_gradients (spinup/utils/mpi_tf.py:45-80: Allreduce(SUM) of the flat
 * gradient, division by the number of processes, Adam, parameter Bcast).  Every rank creates a comm (one device slab: flag
 * words + two halves of max_floats), exports its 64-byte cudaIpcMemHandle_t, the caller gathers the handles of all ranks (any
 * transport) and connects.  No reference counterpart for the plumbing: the reference is MPI on CPUs. */
typedef struct ml4ca_peer_comm ml4ca_peer_comm;
ML4CA_API int ml4ca_peer_comm_create(int32_t rank, int32_t world, int64_t max_floats, int32_t device, ml4ca_peer_comm** out);
ML4CA_API int ml4ca_peer_comm_export(const ml4ca_peer_comm* c, uint8_t* handle64);
/* handles [world][64] in rank order (the own entry is ignored). */
ML4CA_API int ml4ca_peer_comm_connect(ml4ca_peer_comm* c, const uint8_t* handles);
/* The same for ranks that share an address space (several comms in one process: threads as ranks, the single-GPU test of
 * the protocol): slabs [world] = the device pointers ml4ca_peer_comm_slab returned for every rank. */
ML4CA_API int ml4ca_peer_comm_slab(const ml4ca_peer_comm* c, void** slab);
ML4CA_API int ml4ca_peer_comm_connect_ptrs(ml4ca_peer_comm* c, void* const* slabs);
ML4CA_API int ml4ca_peer_comm_destroy(ml4ca_peer_comm* c);
/* steps completed and waits given up (a peer did not publish within 5 s: results of that step are invalid). */
ML4CA_API int ml4ca_peer_comm_status(ml4ca_peer_comm* c, int32_t* steps, int32_t* timeouts);
/* In-place sum over ranks of buf [n] (device), one kernel: publish -> wait -> sum in rank order (bit-identical on every rank).
 * tail_src (nullable, device, double): buf[tail_off + q], q < n_tail, is taken from (float)tail_src[q] (the statistics sums of
 * ml4ca_ppo_grad).  ctl / iter: skipped like ml4ca_ppo_grad_ex.  Every rank must issue the same sequence of calls. */
ML4CA_API int ml4ca_peer_allreduce(ml4ca_peer_comm* c, float* buf, int64_t n, const double* tail_src, int64_t tail_off,
                                   int32_t n_tail, const ml4ca_ppo_ctl* ctl, int32_t iter, void* stream);
/* ml4ca_peer_allreduce of the flat gradient buf [n] (statistics tail of 5 at tail_off) + ml4ca_adam_step_dev on the slice
 * [lo, hi) in the same kernel.  params, m1, m2: bases of the FULL flat vectors (indexed like buf). */
ML4CA_API int ml4ca_adam_step_peer(ml4ca_peer_comm* c, float* buf, int64_t n, const double* tail_src, int64_t tail_off, int64_t lo,
                                   int64_t hi, float* params, float* m1, float* m2, float lr, float beta1, float beta2, float eps,
                                   float grad_scale, int32_t net, int32_t iter, float count, float kl_limit, ml4ca_ppo_ctl* ctl,
                                   void* stream);
/* ml4ca_ppo_grad runs on the tensor cores by default (tcgen05, fp16 operands, fp32 accumulation: gradients to ~1e-3 of
 * the largest component with two hidden layers, 4.5e-3 stated with three) for every network ml4ca_policy_create accepts
 * (64 x 64, 64 x 64 x 64, 80 x 80 x 80).  enable = 1 selects the fp32 CUDA-core kernels (1e-5 .. 2e-4), 0 the tensor-core
 * one, -1 only queries; returns the previous setting.  Initial value: environment variable ML4CA_PPO_FP32. */
ML4CA_API int ml4ca_ppo_use_fp32(int enable);
/* ---- TRPO / NPG pieces (spinup/algos/tf1/trpo/trpo.py:236-247,264-303; trpo/core.py:52-60,88-100) -----------------------------
 * The surrogate pi_loss = -mean(ratio adv) and its flat gradient (trpo.py:237,244) are ml4ca_ppo_grad with net 0 and a
 * clip_ratio large enough never to bind (1e30).  The two passes below run the fp32 CUDA-core kernel unless
 * ml4ca_trpo_use_tensor_cores(1) selects the tcgen05 one.
 * ml4ca_trpo_policy_mu: the distribution "info" the reference's GAEBuffer stores per step (trpo.py:300): mu [T, act_dim, n]
 * of obs [T, obs_dim, n] at the current parameters (log_std is state-independent: the caller copies it from the parameters). */
/* enable = 1 runs the two TRPO passes on the tensor-core gradient kernel (fp16 operands: the Hessian-vector product then needs a
 * wider central-difference bracket and matches the exact one to 0.2-0.3 % instead of 0.02 %, see ml4ca_b200/trpo.py); 0 = the fp32 kernel (default),
 * -1 only queries; returns the previous setting. */
ML4CA_API int ml4ca_trpo_use_tensor_cores(int enable);
ML4CA_API int ml4ca_trpo_policy_mu(ml4ca_policy* p, int64_t n, int32_t T, const float* obs, float* mu, void* stream);
/* d_kl = mean KL(pi_theta || pi_old) (core.diagonal_gaussian_kl as mlp_gaussian_policy calls it, trpo/core.py:52-60,98) over
 * the buffer, and its flat gradient w.r.t. the pi variables and log_std: grad (SUM convention, like ml4ca_ppo_grad; v block
 * zero), stats[2] = sum of per-sample KL, stats[5] = sample count.  mu_old [T, act_dim, n], log_std_old [act_dim] (device).
 * The Hessian-vector product of trpo/core.py:68-72 is a central difference of this gradient (host side, ml4ca_b200/trpo.py). */
ML4CA_API int ml4ca_trpo_kl_grad(ml4ca_policy* p, int64_t n, int32_t T, const float* obs, const float* mu_old,
                                 const float* log_std_old, float* grad, double* stats, void* stream);
/* tf.train.AdamOptimizer step (beta1 0.9, beta2 0.999, eps 1e-8 in the reference) on m parameters:
 * g = grad * grad_scale; m1, m2 moment buffers; t = 1-based step count of this optimizer. */
ML4CA_API int ml4ca_adam_step(int64_t m, float* params, const float* grad, float* m1, float* m2, float lr, float beta1,
                              float beta2, float eps, int32_t t, float grad_scale, void* stream);

ML4CA_API const char* ml4ca_last_error(void);
/* "ml4ca_b200 <version> sm_100a" */
ML4CA_API const char* ml4ca_version(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches evidence) */
ML4CA_API int64_t ml4ca_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* ML4CA_B200_H_ */
