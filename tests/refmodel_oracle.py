"""Float64 NumPy restatement of the DECLARED DP reference model (DESIGN.md section 4, "DP reference model";
csrc/refmodel.cu), the PID with velocity feed-forward, and a float64 closed loop of PID + pseudoinverse on the
stand-in hull (oracle/vessel.py, calm water).

TEST INFRASTRUCTURE, like oracle/: the kernels never import it.

Per env and per DOF (N, E, psi) a third-order reference filter with saturating elements (Fossen 2011, section 12.1):

    eta_d / r = w^3 / ((s + w)(s^2 + 2 zeta w s + w^2))
    jerk      = w^3 e - (2 zeta + 1) w a_d - (2 zeta + 1) w^2 v_d,    e = r - eta_d   (heading: e wrapped to [-pi, pi))

restated as the discrete recurrence the kernel runs: r held over the env step, n_sub = max(1, round(step_dt / SIM_DT))
semi-implicit Euler sub-steps of h = step_dt / n_sub, each

    a_d <- clamp(a_d + h jerk, +-a_max);   v_d <- clamp(v_d + h a_d, +-v_max);   eta_d <- eta_d + h v_d

State rows (the kernel's [9, n] layout): eta_d[0:3], v_d[3:6], a_d[6:9].
"""
import numpy as np

from oracle import constants as C
from oracle import pinv_oracle as PO
from oracle import vessel

# The declared defaults of csrc/ml4ca_constants.h (ML4CA_REF_*), checked by tests/test_refmodel_cpu.py.
REF_ZETA = (1.0, 1.0, 1.0)
REF_OMEGA = (0.2, 0.2, 0.25)          # rad/s
REF_V_MAX = (0.15, 0.1, 0.1)          # m/s, m/s, rad/s
REF_A_MAX = (0.05, 0.02, 0.02)        # m/s^2, m/s^2, rad/s^2
REF_STATE_ROWS = 9

ROWS = REF_STATE_ROWS
ETA, VEL, ACC = slice(0, 3), slice(3, 6), slice(6, 9)


class RefCfg(object):
    """ml4ca_refmodel_cfg; the defaults are ml4ca_refmodel_cfg_default."""

    def __init__(self, step_dt=0.2, zeta=REF_ZETA, omega=REF_OMEGA, v_max=REF_V_MAX, a_max=REF_A_MAX):
        self.step_dt = float(step_dt)
        self.zeta, self.omega, self.v_max, self.a_max = (np.asarray(x, dtype=np.float64).reshape(3)
                                                         for x in (zeta, omega, v_max, a_max))

    @property
    def n_sub(self):
        return max(1, int(np.rint(self.step_dt / C.SIM_DT)))

    @property
    def h(self):
        return self.step_dt / self.n_sub


def wrap(a):
    """a - 2 pi floor((a + pi) / (2 pi)): [-pi, pi)."""
    return a - 2.0 * np.pi * np.floor((a + np.pi) / (2.0 * np.pi))


def reset(eta0):
    """eta_d = eta0 [3, n], v_d = a_d = 0 -> state [9, n]."""
    eta0 = np.asarray(eta0, dtype=np.float64).reshape(3, -1)
    x = np.zeros((ROWS, eta0.shape[1]))
    x[ETA] = eta0
    return x


def step(cfg, state, setpoint, trace=None):
    """One env step of the filter on the held set-point [3, n] -> new state [9, n].  ``trace``: a list that receives the
    state after every sub-step."""
    x = np.array(state, dtype=np.float64).reshape(ROWS, -1)
    r = np.asarray(setpoint, dtype=np.float64).reshape(3, -1)
    h, w, c = cfg.h, cfg.omega[:, None], (2.0 * cfg.zeta + 1.0)[:, None]
    vmax, amax = cfg.v_max[:, None], cfg.a_max[:, None]
    for _ in range(cfg.n_sub):
        e = r - x[ETA]
        e[2] = wrap(e[2])
        jerk = w ** 3 * e - c * w * x[ACC] - c * w ** 2 * x[VEL]
        x[ACC] = np.clip(x[ACC] + h * jerk, -amax, amax)
        x[VEL] = np.clip(x[VEL] + h * x[ACC], -vmax, vmax)
        x[ETA] = x[ETA] + h * x[VEL]
        if trace is not None:
            trace.append(x.copy())
    return x


def substep_matrix(zeta, omega, h):
    """The linear sub-step map z+ = A z of one DOF, z = (eta_d - r, v_d, a_d), limits far away."""
    c = 2.0 * zeta + 1.0
    J = np.array([-omega ** 3, -c * omega ** 2, -c * omega])      # h jerk = h J . z
    a = np.array([0.0, 0.0, 1.0]) + h * J
    v = np.array([0.0, 1.0, 0.0]) + h * a
    x = np.array([1.0, 0.0, 0.0]) + h * v
    return np.stack([x, v, a])


def jury_stable(zeta, omega, h):
    """The stability test ml4ca_refmodel_step applies (include/ml4ca_b200.h): with q = h omega, c = 2 zeta + 1 the
    sub-step map has the characteristic polynomial z^3 + a2 z^2 + a1 z + a0, a2 = q^3 + c q^2 + c q - 3,
    a1 = 3 - 2 c q - c q^2, a0 = c q - 1; its roots lie inside the unit circle iff (Jury) p(1) > 0, p(-1) < 0,
    |a0| < 1 and |a0^2 - 1| > |a0 a2 - a1|."""
    q, c = h * omega, 2.0 * zeta + 1.0
    a2, a1, a0 = q ** 3 + c * q ** 2 + c * q - 3.0, 3.0 - 2.0 * c * q - c * q ** 2, c * q - 1.0
    p1, pm1 = 1.0 + a2 + a1 + a0, -1.0 + a2 - a1 + a0
    return bool(p1 > 0 and pm1 < 0 and abs(a0) < 1 and abs(a0 * a0 - 1.0) > abs(a0 * a2 - a1))


def pid_ff(eta, nu, ref, v_d, integ):
    """oracle/pinv_oracle.pid with velocity feed-forward: the D-term acts on nu - R(psi)^T v_d (v_d NED rates), which is
    pid(eta, nu - R(psi)^T v_d, ref, integ) because nu enters the PID only through Kd nu.  -> (tau, integ)."""
    eta, nu, v_d = (np.asarray(x, dtype=np.float64).reshape(3, -1) for x in (eta, nu, v_d))
    c, s = np.cos(eta[2]), np.sin(eta[2])
    vb = np.stack([c * v_d[0] + s * v_d[1], -s * v_d[0] + c * v_d[1], v_d[2]])
    return PO.pid(eta, nu - vb, ref, integ)


def schedule_at(steps, setpoints, t):
    """s(t): the last entry with steps <= t."""
    k = int(np.searchsorted(np.asarray(steps), t, side="right")) - 1
    return np.asarray(setpoints, dtype=np.float64)[k]


def closed_loop(steps, setpoints, T, cfg=None, dt=0.2):
    """PID (+ velocity feed-forward with a reference model) -> pseudoinverse -> stand-in hull 0 in calm water, one vessel
    starting at rest at s(0), in the step order of evaluate.run_allocator: the PID acts on (eta(t), nu(t), r(t), v_d(t)),
    then the reference advances on s(t), then the hull integrates 20 sub-steps with the allocated thrust.  cfg=None: raw
    set-point steps, r(t) = s(t).  -> dict of float64 arrays eta, ref, setpoint, v_d [T+1, 3] and tau [T, 3]."""
    n_sub = int(np.rint(dt / C.SIM_DT))
    s0 = schedule_at(steps, setpoints, 0).reshape(3, 1)
    eta, nu, integ = s0.copy(), np.zeros((3, 1)), np.zeros((3, 1))
    x = reset(s0) if cfg is not None else None
    rec = {k: np.zeros((T + 1, 3)) for k in ("eta", "ref", "setpoint", "v_d")}
    rec["tau"] = np.zeros((T, 3))
    ref, vd = s0.copy(), np.zeros((3, 1))
    for t in range(T + 1):
        rec["eta"][t], rec["ref"][t], rec["v_d"][t] = eta[:, 0], ref[:, 0], vd[:, 0]
        rec["setpoint"][t] = schedule_at(steps, setpoints, t)
        if t == T:
            break
        tau, integ = pid_ff(eta, nu, ref, vd, integ)
        rec["tau"][t] = tau[:, 0]
        n_pct, alpha = PO.allocate(tau)
        s = rec["setpoint"][t].reshape(3, 1)
        if cfg is not None:
            x = step(cfg, x, s)
            ref, vd = x[ETA].copy(), x[VEL].copy()
        else:
            ref = schedule_at(steps, setpoints, t + 1).reshape(3, 1)
        thrust = np.stack([n_pct[2], n_pct[0], n_pct[1]])                       # env order bow, port, star
        angles = np.stack([np.full_like(alpha[0], C.BOW_ANGLE_FIXED), alpha[0], alpha[1]])
        eta, nu = vessel.integrate(eta, nu, vessel.thruster_wrench(thrust, angles), n_sub)
    return rec


def leg_report(rec, steps, dt=0.2, pos_tol=0.1, yaw_tol_deg=1.0):
    """Per leg k (steps[k] .. steps[k+1], the last entry closes the run): settling time (s, to within pos_tol in N and E
    and yaw_tol in heading, staying there to the end of the leg; inf if never), the largest overshoot past the set-point
    along the leg's move (m for N and E, deg for heading), and the fraction of the leg's steps on which the PID wrench
    is at its saturation in any DOF."""
    sat = np.asarray(C.PID_SAT)
    out = []
    for k in range(len(steps) - 1):
        a, b = int(steps[k]), int(steps[k + 1])
        e = rec["eta"][a:b + 1] - rec["setpoint"][a][None, :]
        e[:, 2] = np.rad2deg(wrap(e[:, 2]))
        ok = (np.abs(e[:, 0]) < pos_tol) & (np.abs(e[:, 1]) < pos_tol) & (np.abs(e[:, 2]) < yaw_tol_deg)
        bad = np.nonzero(~ok)[0]
        settle = 0.0 if bad.size == 0 else (np.inf if bad[-1] == len(ok) - 1 else (bad[-1] + 1) * dt)
        move = rec["setpoint"][a] - (rec["setpoint"][a - 1] if k > 0 else rec["setpoint"][a])
        move[2] = np.rad2deg(move[2])
        over = np.where(move != 0, np.max(np.sign(move)[None, :] * e, axis=0).clip(min=0), 0.0)
        tau = rec["tau"][a:b]
        frac = float(np.mean(np.any(np.abs(tau) >= sat[None, :] - 1e-9, axis=1))) if len(tau) else 0.0
        out.append({"settle_s": settle, "overshoot": over, "saturated": frac})
    return out
