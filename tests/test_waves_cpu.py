"""The declared first-order wave-frequency motion in the float64 oracle (tests/wave_oracle.py): CPU only."""
import numpy as np
import pytest
from scipy import integrate, linalg

import wave_oracle as WO
from oracle import env_oracle as EO

DT = float(np.float32(0.2))


@pytest.mark.parametrize("w0,lam", [(1.0, 0.1), (1.5, 0.05), (2.0, 0.1), (0.3, 0.7), (15.0, 0.1), (3.0, 0.99)])
def test_closed_form_transition_is_the_matrix_exponential(w0, lam):
    """Phi of the underdamped oscillator equals expm(A dt)."""
    np.testing.assert_allclose(WO.transition(w0, lam, DT), linalg.expm(WO.system_matrix(w0, lam) * DT), rtol=0, atol=1e-13)


@pytest.mark.parametrize("w0,lam", [(1.0, 0.1), (2.0, 0.1), (0.3, 0.7), (15.0, 0.1)])
def test_process_noise_is_the_van_loan_integral(w0, lam):
    """Q equals the integral of expm(A s) G G^T expm(A s)^T over [0, dt] with G = [0, sqrt(4 lambda w0^3)] (sigma = 1),
    and Van Loan's block-exponential gives the same matrix."""
    A = WO.system_matrix(w0, lam)
    GGt = np.array([[0.0, 0.0], [0.0, 4.0 * lam * w0 ** 3]])
    quad = np.array([[integrate.quad(lambda s: (linalg.expm(A * s) @ GGt @ linalg.expm(A * s).T)[i, j], 0, DT,
                                     epsabs=1e-13, epsrel=1e-11, limit=200)[0] for j in range(2)] for i in range(2)])
    M = linalg.expm(np.block([[-A, GGt], [np.zeros((2, 2)), A.T]]) * DT)
    van_loan = M[2:, 2:].T @ M[:2, 2:]
    Q = WO.process_noise(w0, lam, DT)
    np.testing.assert_allclose(Q, quad, rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(Q, van_loan, rtol=1e-10, atol=1e-14)
    L = WO.process_noise_factor(w0, lam, DT)
    np.testing.assert_allclose(L @ L.T, Q, rtol=1e-12, atol=1e-15)


def test_stationary_law_is_kept_exactly():
    """Phi P Phi^T + Q = P to 1e-12 over the admissible range (0 < lambda < 1, 0 < w0 dt < pi), for P of any sigma."""
    w0 = np.linspace(0.05, 0.999 * np.pi / DT, 200)
    for lam in (0.01, 0.1, 0.5, 0.95):
        phi, Q = WO.transition(w0, lam, DT), WO.process_noise(w0, lam, DT)
        for sigma in (1.0, 0.2):
            P = WO.stationary_cov(w0, sigma)
            back = np.einsum('ij...,jk...,lk...->il...', phi, P, phi) + sigma * sigma * Q
            assert np.abs(back - P).max() <= 1e-12 * np.abs(P).max()
        L = WO.process_noise_factor(w0, lam, DT)
        assert np.isfinite(L).all() and (L[0, 0] > 0).all() and (L[1, 1] > 0).all()


def test_zero_sigma_gives_zero_motion_and_calm_water():
    """sigma = 0: the reset draws x = x' = 0, the state stays 0, and the measured step is the calm-water step exactly."""
    n, rng = 257, np.random.default_rng(5)
    spec = EO.EnvSpec('final', True, True, max_ep_len=50)
    waves = WO.Waves(sigma=(0.0, 0.0, 0.0), peak_frequency=(1.0, 2.0), damping=0.1, step_dt=DT)
    eta = rng.uniform(-1, 1, (3, n)) * np.array([[5.0], [5.0], [0.5]])
    nu = rng.uniform(-1, 1, (3, n)) * np.array([[0.8], [0.15], [0.3]])
    a_st, b_st = EO.new_state(spec, n), EO.new_state(spec, n)
    oa = EO.reset(spec, a_st, eta=eta, nu=nu)
    ob = WO.reset(spec, b_st, waves, eta=eta, nu=nu, seed=3)
    assert (oa == ob).all() and (b_st['wave'] == 0).all() and (b_st['wave_rate'] == 0).all()
    assert ((b_st['wave_omega'] >= 1.0) & (b_st['wave_omega'] < 2.0)).all()
    for t in range(5):
        act = rng.uniform(-1.2, 1.2, (7, n))
        oa, ra, da, _ = EO.step(spec, a_st, act)
        ob, rb, db, _ = WO.step(spec, b_st, act, waves, seed=3)
        assert (oa == ob).all() and (ra == rb).all() and (da == db).all()
        assert (b_st['wave'] == 0).all() and (b_st['wave_rate'] == 0).all()


def test_oracle_keeps_the_stationary_law():
    """Monte Carlo over the oracle's own Philox draws: the reset draw and 30 steps later have std sigma and w0 sigma
    (within 2 %, 20k envs), and x, x' stay uncorrelated."""
    n = 20000
    waves = WO.Waves(sigma=(0.1, 0.2, 0.05), peak_frequency=(1.0, 1.0), damping=0.1, step_dt=DT)
    ids, word = np.arange(n), np.zeros(n, dtype=np.int64)
    w0, x, xd = waves.sample(7, ids, word)
    assert (w0 == 1.0).all()
    for t in range(31):
        for arr, scale in ((x, waves.sigma), (xd, waves.sigma)):
            assert (np.abs(arr.std(axis=1) / scale - 1) < 0.02).all(), t
        assert (np.abs((x * xd).mean(axis=1)) < 0.03 * waves.sigma ** 2).all()
        word = word + 1
        z1, z2 = WO.DO.normals3(7, ids, word, WO.TAG_STEP1), WO.DO.normals3(7, ids, word, WO.TAG_STEP2)
        x, xd = waves.advance(x, xd, w0, z1, z2)


def test_the_frequency_bound_is_the_nyquist_limit():
    """omega_max * step_dt < pi: at the bound the env-step samples of a motion at w and at 2 pi / dt - w coincide, so the
    observation could not tell them apart; below it the sampled oscillator keeps its own frequency (the eigenvalues of
    Phi have angle w_d dt < pi)."""
    t = np.arange(50) * DT
    w = 0.7 * np.pi / DT
    np.testing.assert_allclose(np.cos(w * t), np.cos((2 * np.pi / DT - w) * t), rtol=0, atol=1e-9)
    for w0 in (0.5, 0.99 * np.pi / DT):
        ev = np.linalg.eigvals(WO.transition(w0, 0.1, DT))
        np.testing.assert_allclose(np.abs(np.angle(ev)), w0 * np.sqrt(1 - 0.01) * DT, rtol=1e-12)
