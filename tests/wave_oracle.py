"""Float64 NumPy restatement of the DECLARED first-order wave-frequency motion (DESIGN.md section 4), built on the env and
disturbance oracles.

TEST INFRASTRUCTURE, like oracle/: the kernels never import it.  It extends oracle/env_oracle.py and
tests/disturbance_oracle.py without changing them.

    per env and DOF d (surge, sway, yaw; body frame):  x'' + 2 lambda w0 x' + w0^2 x = sigma_d sqrt(4 lambda w0^3) w(t)
    stationary law:  P = diag(sigma^2, w0^2 sigma^2)
    exact step over dt:  s <- Phi s + sigma_d L z,  s = [x, x'],  Phi = expm(A dt),  L L^T = Q = P1 - Phi P1 Phi^T
                         (P1 = P with sigma = 1),  z two standard normals per DOF
    measured values:  N + cos(psi) x_s - sin(psi) x_w,  E + sin(psi) x_s + cos(psi) x_w,  psi + x_psi,  nu + x'

Observation, reward and termination are computed from the measured values through EO.observe, EO.reward and
EO.is_terminal; the LF state (eta, nu, the lag, the disturbance) integrates as without waves.

Random numbers: the Philox blocks of tests/disturbance_oracle.py::block, counter word 3 = the stream tags of
csrc/philox.cuh.  A reset draws w0 (tag 5, out0) and the stationary state (tags 6 and 7), keyed by the episode word at
the moment of the reset; every step draws its two normals per DOF (tags 8 and 9) keyed by the word after the step's
increment.
"""
import numpy as np

import disturbance_oracle as DO
from oracle import env_oracle as EO
from oracle import vessel

TAG_OMEGA, TAG_MOTION0, TAG_RATE0, TAG_STEP1, TAG_STEP2 = 5, 6, 7, 8, 9


class Waves(object):
    """ml4ca_env_set_waves: stationary std ``sigma`` (m, m, rad), peak frequency range (rad/s), damping ratio."""

    def __init__(self, sigma=(0.0, 0.0, 0.0), peak_frequency=(1.0, 2.0), damping=0.1, step_dt=0.2):
        self.sigma = np.asarray(sigma, dtype=np.float64)
        self.omega = tuple(float(x) for x in peak_frequency)
        self.damping = float(damping)
        self.step_dt = float(step_dt)

    def sample(self, seed, env_ids, episodes):
        """w0 [n], x [3, n] and x' [3, n] of a new episode (stationary draw)."""
        q = DO.block(seed, env_ids, episodes, TAG_OMEGA)
        w0 = self.omega[0] + (self.omega[1] - self.omega[0]) * DO.unit01(q[0])
        x = self.sigma[:, None] * DO.normals3(seed, env_ids, episodes, TAG_MOTION0)
        xd = w0[None, :] * self.sigma[:, None] * DO.normals3(seed, env_ids, episodes, TAG_RATE0)
        return w0, x, xd

    def advance(self, x, xd, w0, z1, z2):
        """One env step: Phi s + sigma L z per DOF.  x, xd, z1, z2 [3, n]; w0 [n]."""
        phi = transition(w0, self.damping, self.step_dt)
        L = process_noise_factor(w0, self.damping, self.step_dt)
        s = self.sigma[:, None]
        xn = phi[0, 0] * x + phi[0, 1] * xd + s * L[0, 0] * z1
        xdn = phi[1, 0] * x + phi[1, 1] * xd + s * (L[1, 0] * z1 + L[1, 1] * z2)
        return xn, xdn


def system_matrix(w0, lam):
    """A of s' = A s: [[0, 1], [-w0^2, -2 lambda w0]] for one w0."""
    return np.array([[0.0, 1.0], [-w0 * w0, -2.0 * lam * w0]])


def transition(w0, lam, dt):
    """Closed-form Phi = expm(A dt) of the underdamped oscillator, [2, 2, ...] for an array of w0."""
    w0 = np.asarray(w0, dtype=np.float64)
    wd = w0 * np.sqrt(1.0 - lam * lam)
    e = np.exp(-lam * w0 * dt)
    c, s = np.cos(wd * dt), np.sin(wd * dt)
    p12 = e * s / wd
    return np.array([[e * (c + lam * w0 / wd * s), p12], [-w0 * w0 * p12, e * (c - lam * w0 / wd * s)]])


def stationary_cov(w0, sigma=1.0):
    """P = diag(sigma^2, w0^2 sigma^2), [2, 2, ...]."""
    w0 = np.asarray(w0, dtype=np.float64)
    z = np.zeros_like(w0)
    return sigma * sigma * np.array([[1.0 + z, z], [z, w0 * w0]])


def process_noise(w0, lam, dt):
    """Q = P1 - Phi P1 Phi^T (sigma = 1), [2, 2, ...]: the covariance the step must add to stay stationary."""
    phi = transition(w0, lam, dt)
    P = stationary_cov(w0)
    return P - np.einsum('ij...,jk...,lk...->il...', phi, P, phi)


def process_noise_factor(w0, lam, dt):
    """Lower Cholesky factor L of Q, [2, 2, ...]."""
    Q = process_noise(w0, lam, dt)
    l11 = np.sqrt(Q[0, 0])
    l21 = Q[1, 0] / l11
    l22 = np.sqrt(Q[1, 1] - l21 * l21)
    return np.array([[l11, 0 * l11], [l21, l22]])


def measured(eta, nu, x, xd):
    """The measured pose [3, n] and velocity [3, n] from the LF state and the wave motion."""
    eta = np.asarray(eta, dtype=np.float64)
    c, s = np.cos(eta[2]), np.sin(eta[2])
    eta_m = np.stack([eta[0] + c * x[0] - s * x[1], eta[1] + s * x[0] + c * x[1], eta[2] + x[2]])
    return eta_m, np.asarray(nu, dtype=np.float64) + xd


def reset(spec, state, waves, dist=None, mask=None, seed=0, env_id_offset=0, **kw):
    """env_oracle.reset (or disturbance_oracle.reset with ``dist``), then the reset's wave draw (state keys 'wave',
    'wave_rate', 'wave_omega') keyed by the episode word at the moment of the reset.  Returns the measured observation."""
    n = state['ep_len'].shape[0]
    m = np.ones(n, dtype=bool) if mask is None else np.asarray(mask, dtype=bool)
    ids = np.arange(n, dtype=np.int64) + int(env_id_offset)
    w0, x, xd = waves.sample(seed, ids, EO.episode_word(state))
    if dist is None:
        EO.reset(spec, state, mask=mask, seed=seed, env_id_offset=env_id_offset, **kw)
    else:
        DO.reset(spec, state, dist, mask=mask, seed=seed, env_id_offset=env_id_offset, **kw)
    state.setdefault('wave', np.zeros((3, n)))
    state.setdefault('wave_rate', np.zeros((3, n)))
    state.setdefault('wave_omega', np.ones(n))
    state['wave'][:, m], state['wave_rate'][:, m], state['wave_omega'][m] = x[:, m], xd[:, m], w0[m]
    return observe(spec, state)


def observe(spec, state):
    """EO.observe of the measured pose and velocity."""
    eta_m, nu_m = measured(state['eta'], state['nu'], state['wave'], state['wave_rate'])
    return EO.observe(spec, eta_m, nu_m, state['ref'], state['prev_thrust'])


def step(spec, state, action, waves, dist=None, seed=0, env_id_offset=0):
    """One env step: the LF state moves as in env_oracle.step (disturbance_oracle.step with ``dist``), the wave state takes
    one exact step with the normals of (seed, env id, episode word after this step's increment), and observation, reward
    and termination come from the measured values.  Returns (obs, reward, done, info) like env_oracle.step."""
    act, sat = EO.transform_action(spec, action)
    prev_angles = state['angles'].copy()
    thrust = act[0:3]
    for idx in spec.valid:
        if idx >= 3:
            state['angles'][idx - 3] = act[spec.amap[idx]]
    if spec.n_substeps > 0:
        tau = vessel.thruster_wrench(thrust, state['angles'])
        lag = dict(tau_act=state['tau_act'], lag_s=spec.actuator_lag_s) if spec.actuator_lag_s > 0 else {}
        if dist is None:
            out = vessel.integrate(state['eta'], state['nu'], tau, spec.n_substeps, params=spec.hull, **lag)
        else:
            out = DO.step_disturbed(state['eta'], state['nu'], tau, spec.n_substeps, state['current'], state['bias'],
                                    params=spec.hull, **lag)
        if lag:
            state['tau_act'] = out[2]
        state['eta'], state['nu'] = out[0], out[1]
    n = state['ep_len'].shape[0]
    ids = np.arange(n, dtype=np.int64) + int(env_id_offset)
    state['ep_len'] = state['ep_len'] + 1
    word = EO.episode_word(state)
    z1, z2 = DO.normals3(seed, ids, word, TAG_STEP1), DO.normals3(seed, ids, word, TAG_STEP2)
    state['wave'], state['wave_rate'] = waves.advance(state['wave'], state['wave_rate'], state['wave_omega'], z1, z2)
    obs = observe(spec, state)
    old_scaled = obs[6:9] if spec.extended_state else None
    state['prev_thrust'] = thrust.copy()
    rew = EO.reward(spec, obs[0:3], obs[3:6], state['prev_thrust'], old_scaled, state['angles'], prev_angles)
    done = EO.is_terminal(spec, obs)
    truncated = state['ep_len'] >= spec.max_ep_len
    if dist is not None and dist.bias_time_s > 0:
        w = DO.normals3(seed, ids, word, DO.TAG_BIAS_STEP)
        state['bias'] = DO.gauss_markov(state['bias'], dist.a, dist.gain, w)
    return obs, rew, done, {'sat': sat, 'truncated': truncated, 'act': act}
