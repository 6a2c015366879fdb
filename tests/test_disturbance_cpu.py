"""The declared environmental disturbance (ocean current + Gauss-Markov bias force) in the float64 oracle: CPU only."""
import numpy as np

import disturbance_oracle as DO
from oracle import env_oracle as EO
from oracle import philox


def _start(spec, n, rng):
    st = EO.new_state(spec, n)
    eta = rng.uniform(-1, 1, (3, n)) * np.array([[5.0], [5.0], [0.5]])
    nu = rng.uniform(-1, 1, (3, n)) * np.array([[0.8], [0.15], [0.3]])
    EO.reset(spec, st, eta=eta, nu=nu)
    return st


def test_zero_disturbance_is_calm_water_exactly():
    """Zero current and zero bias: the disturbed step is today's step, float64 ==, with and without the wrench lag."""
    n, rng = 257, np.random.default_rng(3)
    for lag in (0.0, 0.92):
        spec = EO.EnvSpec('final', True, True, hull_model=1 if lag else 0, actuator_lag_s=lag)
        dist = DO.Disturbance(bias_time_s=5.0)
        a_st = _start(spec, n, rng)
        b_st = {k: v.copy() for k, v in a_st.items()}
        b_st['current'], b_st['bias'] = np.zeros((2, n)), np.zeros((3, n))
        for t in range(4):
            act = rng.uniform(-1.2, 1.2, (7, n))
            oa, ra, da, _ = EO.step(spec, a_st, act)
            ob, rb, db, _ = DO.step(spec, b_st, act, dist, seed=1)
            assert (oa == ob).all() and (ra == rb).all() and (da == db).all()
            for k in ('eta', 'nu', 'tau_act', 'prev_thrust', 'angles'):
                assert (a_st[k] == b_st[k]).all(), k
            assert (b_st['bias'] == 0).all()


def test_drifting_hull_takes_the_current_velocity():
    """Zero thrust in a current V: the velocity over ground converges to v_c (relative velocity to 0) and the position
    then drifts at V.  The slowest mode is surge, m11 / Xu = 26.4 s for hull model 0: 1e-6 of 0.2 m/s takes ~6 minutes."""
    n = 4
    spec = EO.EnvSpec('full', False, False, max_ep_len=10 ** 6)
    beta = np.array([0.0, np.pi / 2, 2.0, -2.5])
    V = np.array([0.1, 0.2, 0.05, 0.15])
    st = EO.new_state(spec, n)
    EO.reset(spec, st, eta=np.stack([np.zeros(n), np.zeros(n), np.array([0.0, 0.3, -0.2, 0.1])]), nu=np.zeros((3, n)))
    st['current'] = np.stack([V * np.cos(beta), V * np.sin(beta)])
    st['bias'] = np.zeros((3, n))
    dist = DO.Disturbance()
    zero = np.zeros((6, n))
    for _ in range(2000):                                  # 400 s
        DO.step(spec, st, zero, dist)
    ur, vr = DO.rot_t(st['eta'][2], *st['current'])
    assert np.abs(st['nu'][0] - ur).max() < 1e-6 and np.abs(st['nu'][1] - vr).max() < 1e-6
    assert np.abs(st['nu'][2]).max() < 1e-6
    ne0 = st['eta'][:2].copy()
    for _ in range(50):                                    # 10 s
        DO.step(spec, st, zero, dist)
    np.testing.assert_allclose((st['eta'][:2] - ne0) / 10.0, st['current'], rtol=0, atol=1e-6)


def test_gauss_markov_bias_statistics():
    """From its stationary draw, the bias keeps std sigma and has lag-1 autocorrelation a = exp(-step_dt / T_b)."""
    n, seed = 200000, 9
    spec = EO.EnvSpec('final', True, True, n_substeps=0, max_ep_len=10 ** 6)
    sigma = np.array([20.0, 10.0, 5.0])
    dist = DO.Disturbance(bias_std=sigma, bias_time_s=2.0)
    st = EO.new_state(spec, n)
    DO.reset(spec, st, dist, seed=seed)
    act = np.zeros((7, n))
    act[4] = act[6] = 1.0
    prev = st['bias'].copy()
    cs, ss = [], []
    for _ in range(5):
        DO.step(spec, st, act, dist, seed=seed)
        b = st['bias']
        cs.append((prev * b).mean(axis=1) / (prev.std(axis=1) * b.std(axis=1)))
        ss.append(b.std(axis=1))
        prev = b.copy()
    err = 4.0 / np.sqrt(n)                                  # ~4 standard errors
    assert np.abs(np.mean(ss, axis=0) / sigma - 1).max() < 2 * err
    assert np.abs(np.mean(cs, axis=0) - dist.a).max() < 2 * err
    assert abs(dist.a - np.exp(-0.1)) < 1e-15


def test_disturbance_streams_are_new_tags():
    """The current / bias streams use counter words that no earlier stream used; the reset-thrust normals are unchanged."""
    assert {DO.TAG_CURRENT, DO.TAG_BIAS0, DO.TAG_BIAS_STEP}.isdisjoint({DO.TAG_RESET_POSE,
                                                                                     DO.TAG_RESET_THRUST})
    ids, word = np.arange(8), np.full(8, 3 << 16 | 7)
    q = philox.philox4x32(ids, 0, word, 1, 5, 0x5EED5EED)
    r0 = np.sqrt(-2.0 * np.log(philox.unit_open(q[0]).astype(np.float64)))
    a0 = 2.0 * np.pi * (q[1] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    np.testing.assert_array_equal(philox.reset_thrust_normals(5, ids, word)[0], r0 * np.cos(a0))
    # the kernels draw the reset-thrust normals and the bias normals through one Box-Muller routine: the tag alone differs
    np.testing.assert_array_equal(DO.normals3(5, ids, word, DO.TAG_RESET_THRUST), philox.reset_thrust_normals(5, ids, word))
    assert not np.allclose(DO.normals3(5, ids, word, DO.TAG_BIAS0), philox.reset_thrust_normals(5, ids, word))
