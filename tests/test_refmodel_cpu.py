"""The float64 restatement of the DP reference model (tests/refmodel_oracle.py) against its specification: the declared
defines, the transfer function in the linear regime, the limits, the heading wrap, the stability test, and the declared
defaults over the box test in the float64 closed loop.  Plus the box-test schedule and the harness' schedule checks."""
import os
import re

import numpy as np
import pytest
from scipy import signal

import refmodel_oracle as R
from oracle import constants as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def defines():
    out = {}
    for line in open(os.path.join(ROOT, "ml4ca_b200", "csrc", "ml4ca_constants.h")):
        m = re.match(r"#define\s+(ML4CA_REF_\w+)\s+\(?([-0-9.e]+)\)?", line.strip())
        if m:
            out[m.group(1)] = float(m.group(2))
    return out


def test_defines_mirror():
    d = defines()
    for name, want in (("ZETA", R.REF_ZETA), ("OMEGA", R.REF_OMEGA), ("V_MAX", R.REF_V_MAX), ("A_MAX", R.REF_A_MAX)):
        assert tuple(d["ML4CA_REF_%s_%s" % (name, k)] for k in ("N", "E", "PSI")) == want, name
    assert d["ML4CA_REF_STATE_ROWS"] == R.REF_STATE_ROWS


def test_linear_regime_matches_the_transfer_function():
    """Limits far away: the recurrence against scipy.signal.lsim of w^3 / ((s + w)(s^2 + 2 zeta w s + w^2)) for a 1 m step.
    Semi-implicit Euler at h = 0.01 s is first-order accurate: the difference is O(h w) of the step, here below 0.4 %."""
    zeta, w = np.array([1.0, 0.7, 1.3]), np.array([0.2, 0.5, 0.25])
    cfg = R.RefCfg(step_dt=0.2, zeta=zeta, omega=w, v_max=(1e6,) * 3, a_max=(1e6,) * 3)
    T = 400
    x = R.reset(np.zeros(3))
    got = [x[R.ETA, 0].copy()]
    for _ in range(T):
        x = R.step(cfg, x, np.array([1.0, 1.0, 1.0]))
        got.append(x[R.ETA, 0].copy())
    got = np.array(got)
    t = np.arange(T + 1) * 0.2
    for d in range(3):
        num = [w[d] ** 3]
        den = np.polymul([1.0, w[d]], [1.0, 2 * zeta[d] * w[d], w[d] ** 2])
        _, y, _ = signal.lsim((num, den), np.ones_like(t), t)
        assert np.abs(got[:, d] - y).max() < 4e-3, d


def test_converges_to_a_constant_setpoint():
    cfg = R.RefCfg()
    x = R.reset(np.array([[0.0, 2.0], [0.0, -3.0], [0.0, 0.5]]))
    r = np.array([[4.0, -1.0], [-2.0, 1.0], [1.0, -0.3]])
    for _ in range(1500):
        x = R.step(cfg, x, r)
    np.testing.assert_allclose(x[R.ETA], r, atol=1e-9)
    np.testing.assert_allclose(x[R.VEL], 0.0, atol=1e-9)
    np.testing.assert_allclose(x[R.ACC], 0.0, atol=1e-9)


def test_limits_hold_at_every_substep():
    """20 m and 170 deg steps: both limits are reached, and never exceeded, at any sub-step."""
    cfg = R.RefCfg()
    x = R.reset(np.zeros(3))
    trace = []
    for _ in range(600):
        x = R.step(cfg, x, np.array([20.0, -20.0, np.deg2rad(170.0)]), trace=trace)
    tr = np.array(trace)[:, :, 0]
    assert (np.abs(tr[:, R.VEL]) <= cfg.v_max + 1e-15).all() and (np.abs(tr[:, R.ACC]) <= cfg.a_max + 1e-15).all()
    np.testing.assert_allclose(np.abs(tr[:, R.VEL]).max(axis=0), cfg.v_max)
    np.testing.assert_allclose(np.abs(tr[:, R.ACC]).max(axis=0), cfg.a_max)


def test_heading_step_across_pi_takes_the_short_way():
    cfg = R.RefCfg()
    x = R.reset(np.array([0.0, 0.0, np.deg2rad(170.0)]))
    target = np.deg2rad(-170.0)
    path = []
    for _ in range(400):
        x = R.step(cfg, x, np.array([0.0, 0.0, target]))
        path.append(x[2, 0])
    path = np.array(path)
    assert (np.diff(path) >= -1e-12).all()                                   # increasing through +pi, never back
    assert abs(R.wrap(path[-1] - target)) < 1e-6 and abs(path[-1] - np.deg2rad(190.0)) < 1e-6   # not wrapped itself


def test_stability_test_matches_the_spectral_radius():
    for zeta in (0.3, 1.0, 2.0):
        for w in np.geomspace(0.05, 400.0, 60):
            for h in (0.005, 0.01):
                rho = np.abs(np.linalg.eigvals(R.substep_matrix(zeta, w, h))).max()
                if abs(rho - 1.0) > 1e-6:
                    assert R.jury_stable(zeta, w, h) == (rho < 1.0), (zeta, w, h, rho)
    assert R.jury_stable(1.0, 0.25, 0.01) and not R.jury_stable(1.0, 100.0, 0.01)


# Tuning criteria (DESIGN.md section 4): every leg settled to < 0.1 m / 1 deg within its hold, and the PID wrench
# saturated on < 5 % of a leg's steps.  The declared defaults meet the saturation criterion on every leg and the
# settling criterion on every leg but the combined surge + sway one, where the PID's integrator, wound up by the sway
# lag, leaves 0.13 m after 60 s; a slower reference cannot fix that without failing the sway leg's hold (DESIGN.md).
COMBINED_LEG = 4


def test_defaults_over_the_box_test_in_the_float64_closed_loop():
    from ml4ca_b200.evaluate import box_test_schedule
    steps, sp = box_test_schedule()
    raw = R.leg_report(R.closed_loop(steps, sp, int(steps[-1])), steps)
    rec = R.closed_loop(steps, sp, int(steps[-1]), R.RefCfg())
    rep = R.leg_report(rec, steps)
    for k, leg in enumerate(rep):
        assert leg["saturated"] < 0.05, (k, leg)
        if k != COMBINED_LEG:
            assert leg["settle_s"] < 60.0, (k, leg)
    a, b = int(steps[COMBINED_LEG]), int(steps[COMBINED_LEG + 1])
    assert np.abs(rec["eta"][b, 0:2] - sp[COMBINED_LEG, 0:2]).max() < 0.15
    assert max(leg["saturated"] for leg in raw) > 0.3                # raw steps saturate the PID for a third of a leg
    assert (np.abs(rec["v_d"]) <= np.asarray(R.REF_V_MAX) + 1e-12).all()


def test_box_test_schedule_layout():
    from ml4ca_b200.evaluate import box_test_schedule
    steps, sp = box_test_schedule()
    np.testing.assert_array_equal(steps, np.arange(7) * 300)
    y = np.deg2rad(-45.0)
    np.testing.assert_allclose(sp, [[0, 0, 0], [5, 0, 0], [5, 5, 0], [5, 5, y], [0, 5, y], [0, 0, 0], [0, 0, 0]])
    steps, sp = box_test_schedule(side=3.0, yaw_deg=30.0, hold_s=10.0, dt=0.1)
    np.testing.assert_array_equal(steps, np.arange(7) * 100)
    assert sp[3, 2] == pytest.approx(np.deg2rad(30.0)) and sp[2, 1] == 3.0
    assert R.schedule_at(steps, sp, 99)[0] == 0.0 and R.schedule_at(steps, sp, 100)[0] == 3.0


class _FakeEnv(object):
    """Enough of a Revolt for the schedule checks, which all run before the first device call."""
    num_envs, dt, name, max_ep_len = 4, 0.2, "revoltfinal", 400
    device = "cpu"
    _observer = None


class _FakeModel(object):
    def __init__(self, n, dt):
        self.num_envs, self.step_dt = n, dt


@pytest.mark.parametrize("runner", ["rl", "qp"])
def test_schedule_validation_errors(runner):
    from ml4ca_b200 import evaluate
    env = _FakeEnv()

    def run(**kw):
        if runner == "rl":
            return evaluate.run_RL_policy(env, None, **kw)
        return evaluate.run_allocator(env, "qp", **kw)
    good = (np.array([0, 10]), np.zeros((2, 3)))
    with pytest.raises(ValueError):
        run(schedule=(np.array([1, 10]), np.zeros((2, 3))))                   # does not start at 0
    with pytest.raises(ValueError):
        run(schedule=(np.array([0, 10, 10]), np.zeros((3, 3))))               # not strictly increasing
    with pytest.raises(ValueError):
        run(schedule=(np.array([0, 10]), np.zeros((3, 3))))                   # set-points of the wrong length
    with pytest.raises(ValueError):
        run(schedule=good, reference_model=_FakeModel(5, 0.2))                # num_envs mismatch
    with pytest.raises(ValueError):
        run(schedule=good, reference_model=_FakeModel(4, 0.1))                # step_dt mismatch
    with pytest.raises(ValueError):
        run(reference_model=_FakeModel(4, 0.2))                               # a model without a schedule
    if runner == "rl":
        with pytest.raises(ValueError):
            run(schedule=good, new_ref=np.zeros(3), ref_change_at=3)
        with pytest.raises(ValueError):
            run(schedule=good, ref_change_at=3)
