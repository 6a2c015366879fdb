"""Float64 NumPy restatement of the DECLARED passive nonlinear DP observer (DESIGN.md section 4, "DP observer";
csrc/observer.cu), built on oracle/vessel.py for the hull constants and the thruster model.

TEST INFRASTRUCTURE, like oracle/: the kernels never import it.

It restates the discrete recurrence the kernel runs, not the ODE: y, tau and psi_m held over the env step,
n_sub = max(1, round(step_dt / SIM_DT)) semi-implicit Euler sub-steps of h = step_dt / n_sub, the innovation recomputed
every sub-step, velocity-type states (xi2, nu, b) from the old state, then position-type states (xi1, eta) with the new
xi2, nu:

    e     = y - eta - xi2                    (e_psi wrapped: a - 2 pi floor((a + pi) / (2 pi)))
    xi2  <- xi2 + h (-w^2 xi1 - 2 lambda w xi2 + K12 e)
    nu   <- nu + h M^-1 (tau - D(nu) nu - Coriolis(nu) + R(psi_m)^T (b + K4 e))
    b    <- b + h (-b / T_b + K3 e)          (T_b = 0: no decay)
    xi1  <- xi1 + h (xi2_new + K11 e)
    eta  <- eta + h (R(psi_m) nu_new + K2 e)

K11 = -2 (zeta_n - lambda) w_c / w, K12 = 2 w (zeta_n - lambda), K2 = w_c = cutoff_ratio w.  State rows (the kernel's
[15, n] layout): xi1[0:3], xi2[3:6], eta[6:9], nu[9:12], b[12:15].
"""
import numpy as np

from oracle import constants as C
from oracle import vessel

# The declared defaults and limits of csrc/ml4ca_constants.h (ML4CA_OBS_*), checked by tests/test_observer_cpu.py.
OBS_NOTCH_DAMPING = 1.0
OBS_WAVE_DAMPING = 0.1
OBS_CUTOFF_RATIO = 1.2
OBS_BIAS_TIME_S = 0.0
OBS_K4_PER_MASS = 0.2
OBS_K3_PER_K4 = 0.2
OBS_PEAK_FREQUENCY = 1.5
OBS_OMEGA_RANGE = (0.1, 10.0)
OBS_STATE_ROWS = 15

ROWS = OBS_STATE_ROWS
XI1, XI2, ETA, NU, BIAS = slice(0, 3), slice(3, 6), slice(6, 9), slice(9, 12), slice(12, 15)


class ObserverCfg(object):
    """ml4ca_observer_cfg; the defaults are ml4ca_observer_cfg_default(hull_model)."""

    def __init__(self, hull_model=0, step_dt=0.2, notch_damping=OBS_NOTCH_DAMPING, wave_damping=OBS_WAVE_DAMPING,
                 cutoff_ratio=OBS_CUTOFF_RATIO, bias_time_s=OBS_BIAS_TIME_S, k3=None, k4=None):
        p = C.HULL_MODELS[hull_model]
        m = np.array([p['m11'], p['m22'], p['m33']])
        self.hull_model = int(hull_model)
        self.params = p
        self.step_dt = float(step_dt)
        self.zeta = float(notch_damping)
        self.lam = float(wave_damping)
        self.cutoff = float(cutoff_ratio)
        self.bias_time_s = float(bias_time_s)
        self.k4 = OBS_K4_PER_MASS * m if k4 is None else np.asarray(k4, dtype=np.float64)
        self.k3 = OBS_K3_PER_K4 * self.k4 if k3 is None else np.asarray(k3, dtype=np.float64)

    @property
    def n_sub(self):
        return max(1, int(np.rint(self.step_dt / C.SIM_DT)))

    def gains(self, w):
        """(K11, K12, K2) for peak frequency w (scalar or array)."""
        w = np.asarray(w, dtype=np.float64)
        wc = self.cutoff * w
        return -2.0 * (self.zeta - self.lam) * wc / w, 2.0 * w * (self.zeta - self.lam), wc


def wrap(a):
    """a - 2 pi floor((a + pi) / (2 pi)): [-pi, pi)."""
    return a - 2.0 * np.pi * np.floor((a + np.pi) / (2.0 * np.pi))


def clamp_omega(w):
    """The kernel's treatment of w_o: clamped into OBS_OMEGA_RANGE, NaN -> the lower bound."""
    lo, hi = OBS_OMEGA_RANGE
    w = np.asarray(w, dtype=np.float64)
    return np.clip(np.where(np.isnan(w), lo, w), lo, hi)


def reset(y):
    """State [15, n] of a reset from y [3, n]."""
    y = np.asarray(y, dtype=np.float64)
    x = np.zeros((ROWS,) + y.shape[1:])
    x[ETA] = y
    return x


def step_tau(cfg, x, y, tau, omega):
    """One env step from the body-frame wrench tau [3, n].  x [15, n] (not modified), y [3, n], omega [n] -> new x."""
    x = np.array(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    tau = np.asarray(tau, dtype=np.float64)
    w = clamp_omega(omega)
    k11, k12, k2 = cfg.gains(w)
    p = cfg.params
    m11, m22, m33 = p['m11'], p['m22'], p['m33']
    n_sub = cfg.n_sub
    h = cfg.step_dt / n_sub
    inv_tb = 1.0 / cfg.bias_time_s if cfg.bias_time_s > 0 else 0.0
    k3, k4 = cfg.k3[:, None], cfg.k4[:, None]
    c, s = np.cos(y[2]), np.sin(y[2])
    xi1, xi2, eta, nu, b = x[XI1], x[XI2], x[ETA], x[NU], x[BIAS]
    for _ in range(n_sub):
        e = y - eta - xi2
        e = np.stack([e[0], e[1], wrap(e[2])])
        xi2n = xi2 + h * (-w * w * xi1 - 2.0 * cfg.lam * w * xi2 + k12 * e)
        g = b + k4 * e
        fx, fy, fn = c * g[0] + s * g[1], c * g[1] - s * g[0], g[2]
        u, v, r = nu
        du = (tau[0] + fx + m22 * v * r - (p['Xu'] + p['Xuu'] * np.abs(u)) * u) / m11
        dv = (tau[1] + fy - m11 * u * r - (p['Yv'] + p['Yvv'] * np.abs(v)) * v) / m22
        dr = (tau[2] + fn - (m22 - m11) * u * v - (p['Nr'] + p['Nrr'] * np.abs(r)) * r) / m33
        nun = np.stack([u + h * du, v + h * dv, r + h * dr])
        b = b + h * (-inv_tb * b + k3 * e)
        xi1 = xi1 + h * (xi2n + k11 * e)
        eta = eta + h * (np.stack([c * nun[0] - s * nun[1], s * nun[0] + c * nun[1], nun[2]]) + k2 * e)
        xi2, nu = xi2n, nun
    return np.concatenate([xi1, xi2, eta, nu, b])


def step(cfg, x, y, thrust, angles, omega, restart=None):
    """ml4ca_observer_step: thrust [3, n] (%), angles [3, n] (rad), env order bow, port, star; restart [n] (nullable)."""
    out = step_tau(cfg, x, y, vessel.thruster_wrench(thrust, angles), omega)
    if restart is not None:
        m = np.asarray(restart) != 0
        out[:, m] = reset(np.asarray(y, dtype=np.float64)[:, m])
    return out


def one_step_map(cfg, omega, psi, hull_nu=None, eps=1e-6):
    """The numerically linearised one-step map of the error dynamics at nu^ = 0 (or ``hull_nu``), heading psi, for one env:
    (A [15, 15], B [15, 3]) with x+ = A x + B y about the zero state and zero input (tau = 0), by central differences.
    The observer is driven only by y and tau, so the estimation error of a true LF system obeys the same A."""
    x0 = np.zeros((ROWS, 1))
    if hull_nu is not None:
        x0[NU, 0] = hull_nu
    y0 = np.array([[0.0], [0.0], [psi]])
    x0[ETA, 0] = y0[:, 0]
    tau = np.zeros((3, 1))
    om = np.array([omega])
    A = np.empty((ROWS, ROWS))
    B = np.empty((ROWS, 3))
    for j in range(ROWS):
        d = np.zeros((ROWS, 1))
        d[j] = eps
        A[:, j] = (step_tau(cfg, x0 + d, y0, tau, om) - step_tau(cfg, x0 - d, y0, tau, om))[:, 0] / (2 * eps)
    for j in range(3):
        d = np.zeros((3, 1))
        d[j] = eps
        B[:, j] = (step_tau(cfg, x0, y0 + d, tau, om) - step_tau(cfg, x0, y0 - d, tau, om))[:, 0] / (2 * eps)
    return A, B


def frequency_response(A, B, w, dt, out_rows=ETA):
    """|H(e^{j w dt})| of the discrete map x+ = A x + B y to the rows ``out_rows``: [len(w), rows, 3]."""
    I = np.eye(A.shape[0])
    Cm = I[out_rows]
    H = [Cm @ np.linalg.solve(np.exp(1j * wk * dt) * I - A, B) for wk in np.atleast_1d(w)]
    return np.abs(np.array(H))
