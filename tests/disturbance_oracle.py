"""Float64 NumPy restatement of the DECLARED environmental disturbance (DESIGN.md section 4), built on the env oracle.

TEST INFRASTRUCTURE, like oracle/: the kernels never import it.  It extends oracle/vessel.py and oracle/env_oracle.py
without changing them, so that their calm-water behaviour stays what the golden vectors pin.

    ocean current, constant in NED over an episode:   v_c = V [cos beta, sin beta],  V ~ U(speed range),
                                                       beta ~ U(direction range), the direction the water flows towards
    relative velocity (Fossen, irrotational constant current):   nu_r = nu - R(psi)^T [v_cN, v_cE, 0]^T
    the hull equations of oracle/vessel.py act on nu_r;  eta_dot = R(psi) nu_r + [v_cN, v_cE, 0]^T
    bias force b = [X_N, Y_E, N_psi] in NED, first-order Gauss-Markov per env step:
        b <- a b + sigma sqrt(1 - a^2) w,  a = exp(-step_dt / T_b)  (T_b = 0: a = 1),  w ~ N(0, I);  at a reset b = sigma w0

One env step (step_disturbed): nu -> nu_r with the heading at the start of the step; the sub-steps of vessel.integrate on
nu_r with the body-frame force R(psi0)^T b added to the (lagged) thruster wrench and held; N, E += n_sub h v_c; nu_r -> nu
with the heading at the end of the step.  The Gauss-Markov update of b follows the sub-steps.

Random numbers: Philox4x32-10 of oracle/philox.py keyed by (seed, global env id, episode word), counter word 3 = the stream
tag of csrc/philox.cuh.
"""
import numpy as np

from oracle import constants as C
from oracle import env_oracle as EO
from oracle import philox
from oracle import vessel

# Counter word 3 of every stream (csrc/philox.cuh): one tag per stream of an (env, episode word).
TAG_RESET_POSE, TAG_RESET_THRUST, TAG_CURRENT, TAG_BIAS0, TAG_BIAS_STEP = 0, 1, 2, 3, 4


def block(seed, env_id, episode, tag):
    """The Philox block of (env, episode word, tag): counter (env_lo, env_hi, word, tag), key (seed_lo,
    seed_hi ^ 0x5EED5EED).  Returns 4 uint32 arrays."""
    env_id = np.asarray(env_id, dtype=np.uint64)
    episode = np.asarray(episode, dtype=np.uint64)
    k0 = int(seed) & 0xFFFFFFFF
    k1 = ((int(seed) >> 32) & 0xFFFFFFFF) ^ 0x5EED5EED
    lo = env_id & np.uint64(0xFFFFFFFF)
    hi = env_id >> np.uint64(32)
    return philox.philox4x32(lo, hi, episode & np.uint64(0xFFFFFFFF), np.full_like(lo, int(tag)), k0, k1)


def unit01(x):
    """uint32 -> [0, 1):  (x >> 8) * 2^-24 (exact in float32 and float64)."""
    return (np.asarray(x, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def current_units(seed, env_id, episode):
    """The two uniforms of a new episode's current (csrc/env_math.cuh::sample_current): speed from out0, direction from
    out1 of the TAG_CURRENT block.  float64 [2, n] in [0, 1)."""
    q = block(seed, env_id, episode, TAG_CURRENT)
    return np.stack([unit01(q[0]), unit01(q[1])])


def normals3(seed, env_id, episode, tag):
    """Three standard normals of the block (env, episode word, tag), as csrc/env_math.cuh::philox_normals3: Box-Muller on
    (out0, out1) -> r0 cos, r0 sin and on (out2, out3) -> r1 cos, r = sqrt(-2 ln unit_open(.)), angle = 2 pi (. >> 8) 2^-24.
    float64 here (the kernel's logf / sincospif are fp32: ~1e-6 relative agreement).  [3, n]"""
    q = block(seed, env_id, episode, tag)
    r0 = np.sqrt(-2.0 * np.log(philox.unit_open(q[0]).astype(np.float64)))
    r1 = np.sqrt(-2.0 * np.log(philox.unit_open(q[2]).astype(np.float64)))
    a0 = 2.0 * np.pi * (q[1] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    a1 = 2.0 * np.pi * (q[3] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    return np.stack([r0 * np.cos(a0), r0 * np.sin(a0), r1 * np.cos(a1)])


class Disturbance(object):
    """ml4ca_env_set_disturbance: ranges of the per-episode current (m/s; rad towards which the water flows), bias force std
    (N, N, Nm) and time constant (s; 0 = constant over the episode)."""

    def __init__(self, current_speed=(0.0, 0.0), current_direction=(0.0, 2 * np.pi), bias_std=(0.0, 0.0, 0.0),
                 bias_time_s=0.0, step_dt=0.2):
        self.speed = tuple(float(x) for x in current_speed)
        self.direction = tuple(float(x) for x in current_direction)
        self.bias_std = np.asarray(bias_std, dtype=np.float64)
        self.bias_time_s = float(bias_time_s)
        self.a = float(np.exp(-step_dt / self.bias_time_s)) if self.bias_time_s > 0 else 1.0
        self.gain = self.bias_std * np.sqrt(1.0 - self.a * self.a)

    def sample(self, seed, env_ids, episodes):
        """Current [2, n] (NED) and bias [3, n] of a new episode, from the Philox streams of (env, episode word)."""
        u = current_units(seed, env_ids, episodes)
        V = self.speed[0] + (self.speed[1] - self.speed[0]) * u[0]
        beta = self.direction[0] + (self.direction[1] - self.direction[0]) * u[1]
        cur = np.stack([V * np.cos(beta), V * np.sin(beta)])
        return cur, self.bias_std[:, None] * normals3(seed, env_ids, episodes, TAG_BIAS0)


def rot_t(psi, xN, yE):
    """R(psi)^T [xN, yE]: NED -> body frame."""
    c, s = np.cos(psi), np.sin(psi)
    return c * xN + s * yE, -s * xN + c * yE


def integrate_force(eta, nu, tau, n_sub, force, h=C.SIM_DT, params=None, tau_act=None, lag_s=0.0):
    """vessel.integrate with a body-frame ``force`` [3, ...] added to the (lagged) wrench at every sub-step, itself not
    lagged.  Same equations and order as vessel.integrate; same returns."""
    p = C.HULL_MODELS[0] if params is None else params
    m11, m22, m33 = p['m11'], p['m22'], p['m33']
    N, E, psi = (np.array(x, dtype=np.float64) for x in eta)
    u, v, r = (np.array(x, dtype=np.float64) for x in nu)
    cmd = np.stack([np.asarray(x, dtype=np.float64) for x in tau])
    f = np.stack([np.asarray(x, dtype=np.float64) for x in force])
    lagged = tau_act is not None
    act = np.array(tau_act, dtype=np.float64) if lagged else cmd
    k = h / (lag_s + h) if lag_s > 0 else 1.0
    for _ in range(int(n_sub)):
        if lagged:
            act = act + k * (cmd - act)
        tx, ty, tn = act + f
        du = (tx + m22 * v * r - (p['Xu'] + p['Xuu'] * np.abs(u)) * u) / m11
        dv = (ty - m11 * u * r - (p['Yv'] + p['Yvv'] * np.abs(v)) * v) / m22
        dr = (tn - (m22 - m11) * u * v - (p['Nr'] + p['Nrr'] * np.abs(r)) * r) / m33
        u = u + h * du
        v = v + h * dv
        r = r + h * dr
        c, s = np.cos(psi), np.sin(psi)
        N = N + h * (c * u - s * v)
        E = E + h * (s * u + c * v)
        psi = psi + h * r
    if lagged:
        return np.stack([N, E, psi]), np.stack([u, v, r]), act
    return np.stack([N, E, psi]), np.stack([u, v, r])


def step_disturbed(eta, nu, tau, n_sub, current, bias, h=C.SIM_DT, params=None, tau_act=None, lag_s=0.0):
    """One env step in ``current`` [2, ...] (NED, m/s) under ``bias`` [3, ...] (NED; N, N, Nm), both held over the step.
    nu in and out is the velocity over ground.  Same returns as vessel.integrate."""
    eta = np.array(eta, dtype=np.float64)
    nu = np.array(nu, dtype=np.float64)
    cN, cE = (np.asarray(x, dtype=np.float64) for x in current)
    bN, bE, bP = (np.asarray(x, dtype=np.float64) for x in bias)
    du, dv = rot_t(eta[2], cN, cE)
    nu_r = np.stack([nu[0] - du, nu[1] - dv, nu[2]])
    fx, fy = rot_t(eta[2], bN, bE)
    out = integrate_force(eta, nu_r, tau, n_sub, np.stack([fx, fy, np.broadcast_to(bP, fx.shape)]), h=h, params=params,
                          tau_act=tau_act, lag_s=lag_s)
    eta1, nu1 = out[0].copy(), out[1].copy()
    eta1[0] = eta1[0] + n_sub * h * cN
    eta1[1] = eta1[1] + n_sub * h * cE
    du, dv = rot_t(eta1[2], cN, cE)
    nu1[0], nu1[1] = nu1[0] + du, nu1[1] + dv
    return (eta1, nu1) + tuple(out[2:])


def gauss_markov(bias, a, gain, w):
    """One env step of the bias: a b + gain w, gain = sigma sqrt(1 - a^2) [3], w [3, ...] standard normals."""
    b = np.asarray(bias, dtype=np.float64)
    g = np.asarray(gain, dtype=np.float64).reshape((3,) + (1,) * (b.ndim - 1))
    return a * b + g * np.asarray(w, dtype=np.float64)


def reset(spec, state, dist, mask=None, seed=0, env_id_offset=0, **kw):
    """env_oracle.reset, then the reset's draw of the current and bias (state keys 'current', 'bias') for the reset envs,
    keyed by the episode word at the moment of the reset."""
    n = state['ep_len'].shape[0]
    m = np.ones(n, dtype=bool) if mask is None else np.asarray(mask, dtype=bool)
    ids = np.arange(n, dtype=np.int64) + int(env_id_offset)
    cur, bias = dist.sample(seed, ids, EO.episode_word(state))
    obs = EO.reset(spec, state, mask=mask, seed=seed, env_id_offset=env_id_offset, **kw)
    state.setdefault('current', np.zeros((2, n)))
    state.setdefault('bias', np.zeros((3, n)))
    state['current'][:, m], state['bias'][:, m] = cur[:, m], bias[:, m]
    return obs


def step(spec, state, action, dist, seed=0, env_id_offset=0, dt=np.float64):
    """env_oracle.step with the hull moving in state['current'] under state['bias'] (step_disturbed); the bias then takes
    one Gauss-Markov step with the normals of (seed, env id, episode word after this step's increment)."""
    act, sat = EO.transform_action(spec, action, dt)
    prev_angles = state['angles'].copy()
    thrust = act[0:3]
    for idx in spec.valid:
        if idx >= 3:
            state['angles'][idx - 3] = act[spec.amap[idx]]
    if spec.n_substeps > 0:
        tau = vessel.thruster_wrench(thrust, state['angles'])
        lag = dict(tau_act=state['tau_act'], lag_s=spec.actuator_lag_s) if spec.actuator_lag_s > 0 else {}
        out = step_disturbed(state['eta'], state['nu'], tau, spec.n_substeps, state['current'], state['bias'],
                             params=spec.hull, **lag)
        if lag:
            state['tau_act'] = out[2]
        state['eta'], state['nu'] = out[0].astype(dt), out[1].astype(dt)
    obs = EO.observe(spec, state['eta'], state['nu'], state['ref'], state['prev_thrust'], dt)
    old_scaled = obs[6:9] if spec.extended_state else None
    state['prev_thrust'] = thrust.astype(dt).copy()
    rew = EO.reward(spec, obs[0:3], obs[3:6], state['prev_thrust'], old_scaled, state['angles'], prev_angles, dt)
    done = EO.is_terminal(spec, obs, dt)
    state['ep_len'] = state['ep_len'] + 1
    truncated = state['ep_len'] >= spec.max_ep_len
    if dist.bias_time_s > 0:                                           # b's value at the start of the step was applied
        ids = np.arange(state['ep_len'].shape[0], dtype=np.int64) + int(env_id_offset)
        w = normals3(seed, ids, EO.episode_word(state), TAG_BIAS_STEP)
        state['bias'] = gauss_markov(state['bias'], dist.a, dist.gain, w)
    return obs, rew, done, {'sat': sat, 'truncated': truncated, 'act': act}
