"""NumPy restatement of the thesis' evaluation metrics (results/all_plots of the reference).

TEST INFRASTRUCTURE (see oracle/__init__.py).
  iae   common.py:57-74 (absolute_error, IAE) with the scaling of box_test/plot_pos.py:174 -- pinned against the
        reference's own common.IAE in tests/test_oracle_pinning.py (matplotlib stubbed)
  work  box_test/plot_act.py:128-135,184-207 (script, not importable: restated)
  iadc  box_test/plot_act.py:320-391 (script: restated)
"""
import numpy as np

RPS_MAX = {'bow': 33.0, 'stern': 11.0}
DIAM = {'bow': 0.06, 'stern': 0.15}
KQ_0 = {'bow': 0.02, 'stern': 0.036}
RHO = 1025.0


def iae(eta, ref, dt):
    """eta [T, 3] (N, E, yaw rad), ref [3] or, for a set-point that changes during the run, [T, 3] (the set-point of each
    sample, as common.py takes it) -> final cumulative IAE with eta, ref / [5, 5, 25 deg]."""
    sc = np.array([5.0, 5.0, 25.0])
    e = np.array(eta, dtype=np.float64).copy()
    r = np.broadcast_to(np.asarray(ref, dtype=np.float64), e.shape).copy()
    e[:, 2], r[:, 2] = np.rad2deg(e[:, 2]), np.rad2deg(r[:, 2])
    err = np.sqrt((((e - r) / sc) ** 2).sum(axis=1))
    return float(((err[1:] + err[:-1]) / 2 * dt).sum())


def power(n, which):
    return np.sign(n) * KQ_0[which] * 2 * np.pi * RHO * DIAM[which] ** 5 * (n / 100.0 * RPS_MAX[which]) ** 3


def work(thrust, dt):
    """thrust [T, 3] (bow, port, star in %) -> W* = trapezoidal integral of the three propeller powers."""
    t = np.asarray(thrust, dtype=np.float64)
    p = np.abs(power(t[:, 0], 'bow')) + np.abs(power(t[:, 1], 'stern')) + np.abs(power(t[:, 2], 'stern'))
    return float(((p[1:] + p[:-1]) / 2 * dt).sum())


def iadc(thrust, angles):
    """thrust [T, 3] %, angles [T, 2] rad -> sum over steps of clip(sum |dn| / 100 + sum |wrap(da_deg)| / 180, 0, 400)."""
    t, a = np.asarray(thrust, dtype=np.float64), np.rad2deg(np.asarray(angles, dtype=np.float64))
    dn = np.abs(np.diff(t, axis=0)).sum(axis=1) / 100.0
    da = np.abs(np.mod(np.diff(a, axis=0) + 180.0, 360.0) - 180.0).sum(axis=1) / 180.0
    return float(np.clip(dn + da, 0, 400).sum())
