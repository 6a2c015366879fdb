"""GPU checks of the first-order wave-frequency motion (ml4ca_env_set_waves): the WAVE variants of the env-step kernel,
the draws of the resets, the measured observation and the Python surface, against the float64 restatement
(tests/wave_oracle.py).

Tolerances are those of tests/test_env_gpu.py and tests/test_disturbance_gpu.py: observation <= 5e-5, reward <= 2e-4,
hull state 2e-5 (position) / 2e-6 (velocity).  The wave state is compared relative to its scale: motion x within
2e-5 sigma and rate x' within 2e-5 w0 sigma after one step from the same state (fp32 Phi, L and Box-Muller normals
against float64; the diagonal of Q is O((w0 dt)^3), so L carries a few 1e-6 relative error), the reset's stationary
draw within 2e-6 of the same scales, and w0 to 1 ulp.  The env's max_ep_len is in the reference's units: max_ep_len = L
gives episodes of L / 2 steps (customEnv.py:83)."""
import ctypes

import numpy as np
import pytest
import torch

import disturbance_oracle as DO
import wave_oracle as WO
from conftest import golden
from oracle import env_oracle as EO

pytestmark = pytest.mark.gpu

TWO_PI = 2 * np.pi
DT = float(np.float32(0.2))
ERR_INVALID = -1                       # ML4CA_ERR_INVALID
SEA = dict(sigma=(0.1, 0.1, np.deg2rad(2.0)), peak_frequency=(1.0, 2.0), damping=0.1)


def make_env(n, kind='final', cont=True, ext=True, hull_kw=None, **kw):
    import ml4ca_b200.env as E
    hull = E.StandInHull(**(hull_kw or {}))
    if kind == 'limited':
        return E.RevoltLimited(hull, extended_state=ext, num_envs=n, **kw)
    return E.RevoltFinal(hull, extended_state=ext, cont_ang=cont, num_envs=n, **kw)


def init_kw(eta, nu):
    z = 0 * eta[0]
    return {'Hull.PosNED': eta[:2], 'Hull.PosAttitude': np.stack([z, z, eta[2]]),
            'Hull.VelocityNu': np.stack([nu[0], nu[1], z, z, z, nu[2]])}


def start_pose(rng, n):
    eta = rng.uniform(-1, 1, (3, n)) * np.array([[4.0], [4.0], [0.4]])
    nu = rng.uniform(-1, 1, (3, n)) * np.array([[0.5], [0.1], [0.2]])
    return eta.astype(np.float32).astype(np.float64), nu.astype(np.float32).astype(np.float64)


def np_(t):
    return t.cpu().numpy()


def ulp_diff(a, b):
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


ZERO_CASES = [('limited', False, False, None, False, True), ('limited', False, True, 0.92, False, True),
              ('final', True, True, None, False, True), ('final', True, True, 0.92, False, True),
              ('limited', False, False, None, True, True), ('final', True, True, 0.92, True, False)]


@pytest.mark.parametrize("kind,cont,ext,lag,dist,exact", ZERO_CASES)
def test_zero_amplitude_waves_equal_calm_water(cuda_device, kind, cont, ext, lag, dist, exact):
    """sigma = 0: the WAVE kernel returns what the default dispatch returns (the WAVE + DIST kernel what the DIST kernel
    returns), over 500 steps with episode-length cuts, terminations and in-kernel restarts (n odd: one env per thread).
    The kernels are compiled separately, and outside the correctly rounded (_rn) operations the compiler is free to form
    multiply-adds differently in each, so bit-for-bit equality is asserted where it holds on the B200 build (every case
    but WAVE + DIST with the lag); there the comparison is at fp32 level on the envs whose flags have agreed so far."""
    n, act_dim = 4099, (7 if cont else 5)
    hull_kw = None if lag is None else dict(hull_model=1, actuator_lag_s=lag)
    kw = dict(seed=4, auto_reset=True, max_ep_len=60, reset_acts=True, device=cuda_device)
    A, B = make_env(n, kind, cont, ext, hull_kw, **kw), make_env(n, kind, cont, ext, hull_kw, **kw)
    if dist:
        for e in (A, B):
            e.set_disturbance(current_speed=(0.0, 0.1), current_direction=(0.0, TWO_PI), bias_std=(5.0, 5.0, 2.0),
                              bias_time_s=3.0)
    B.set_waves(sigma=(0.0, 0.0, 0.0), peak_frequency=(1.0, 2.0), damping=0.1)
    oA, oB = A.reset(), B.reset()
    assert torch.equal(oA, oB)
    g = torch.Generator(device=cuda_device)
    g.manual_seed(1)
    restarts = 0
    sync = torch.ones(n, dtype=torch.bool, device=cuda_device)
    for t in range(500):
        a = torch.rand(act_dim, n, device=cuda_device, generator=g) * 2.4 - 1.2
        oA, rA, _, iA = A.step(a)
        oB, rB, _, iB = B.step(a)
        restarts += int((iA['flags'] != 0).sum())
        if exact:
            assert torch.equal(oA, oB) and torch.equal(rA, rB) and torch.equal(iA['flags'], iB['flags']), t
        sync &= iA['flags'] == iB['flags']
        assert float((oA - oB)[:, sync].abs().max()) <= 1e-4 and float((rA - rB)[sync].abs().max()) <= 5e-4, t
        if t % 50 == 49:
            sA, sB = A.get_state(), B.get_state()
            for k in ("eta", "nu", "prev_thrust", "angles", "ep_len") + (("current", "bias") if dist else ()):
                assert torch.equal(sA[k], sB[k]) if exact else float((sA[k] - sB[k])[..., sync].abs().max()) <= 1e-3, (t, k)
            assert (sB["wave"] == 0).all() and (sB["wave_rate"] == 0).all()
            assert torch.equal(sB["eta_measured"], sB["eta"]) and torch.equal(sB["nu_measured"], sB["nu"])
    assert restarts > n and float(sync.float().mean()) > 0.99


def test_waves_do_not_move_the_hull(cuda_device):
    """With sigma > 0 and the same open-loop actions the LF state (eta, nu, prev_thrust, angles, ep_len) equals that of a
    twin with sigma = 0 bit for bit, and that of a calm twin at fp32 level, on the envs whose flags have agreed so far
    (termination sees the measured values, so waves may end an episode earlier).  set_waves(None) right after a reset
    steps bit for bit like a twin that never had waves.  Gentle actions and a mild sea keep most envs' flags in
    step."""
    n = 4099
    kw = dict(seed=6, auto_reset=True, max_ep_len=80, device=cuda_device)
    mild = dict(sigma=(0.03, 0.03, np.deg2rad(1.0)), peak_frequency=(1.0, 2.0), damping=0.1)
    W, Z, C = make_env(n, **kw), make_env(n, **kw), make_env(n, **kw)
    W.set_waves(**mild)
    Z.set_waves(sigma=(0.0, 0.0, 0.0), peak_frequency=(1.0, 2.0), damping=0.1)
    for e in (W, Z, C):
        e.reset()
    g = torch.Generator(device=cuda_device)
    g.manual_seed(3)
    sync = torch.ones(n, dtype=torch.bool, device=cuda_device)
    moved = 0.0
    restarts = 0
    for t in range(200):
        a = torch.rand(7, n, device=cuda_device, generator=g) * 0.6 - 0.3
        oW, _, _, iW = W.step(a)
        oZ, _, _, iZ = Z.step(a)
        _, _, _, iC = C.step(a)
        sync &= (iW['flags'] == iZ['flags']) & (iW['flags'] == iC['flags'])
        restarts += int((iZ['flags'][sync] != 0).sum())
        moved = max(moved, float((oW - oZ)[:6, sync].abs().max()))
        if t % 30 == 29:
            sW, sZ, sC = W.get_state(), Z.get_state(), C.get_state()
            for k in ("eta", "nu", "prev_thrust", "angles", "ep_len"):
                assert torch.equal(sW[k][..., sync], sZ[k][..., sync]), (t, k)
                assert float((sW[k] - sC[k])[..., sync].abs().max()) <= 1e-3, (t, k)
    assert float(sync.float().mean()) > 0.3 and restarts > n and moved > 0.005   # cuts happened; the observations saw waves
    A, B = make_env(n, **kw), make_env(n, **kw)
    A.set_waves(**SEA)
    A.reset(), B.reset()
    A.set_waves(None)
    assert "wave" not in A.get_state()
    for t in range(60):
        a = torch.rand(7, n, device=cuda_device, generator=g) * 2.0 - 1.0
        oA, rA, _, iA = A.step(a)
        oB, rB, _, iB = B.step(a)
        assert torch.equal(oA, oB) and torch.equal(rA, rB) and torch.equal(iA['flags'], iB['flags']), t


@pytest.mark.parametrize("hull_model,lag,dist", [(0, 0.0, False), (0, 0.0, True), (1, 0.92, False), (1, 0.92, True),
                                                 (0, 0.92, False), (1, 0.0, True)])
def test_wave_step_matches_oracle(cuda_device, hull_model, lag, dist):
    """One step at a time against the float64 oracle: the LF state, the measured observation, reward and done, the wave
    state and w0, through episode-length cuts and in-kernel restarts (which draw a new w0 and a stationary state)."""
    n, seed, L = 2053, 12, 4
    dist_kw = dict(current_speed=(0.0, 0.2), current_direction=(-np.pi, np.pi), bias_std=(15.0, 10.0, 8.0), bias_time_s=4.0)
    spec = EO.EnvSpec('final', True, True, max_ep_len=L, hull_model=hull_model, actuator_lag_s=lag)
    waves = WO.Waves(step_dt=DT, **SEA)
    dO = DO.Disturbance(step_dt=DT, **dist_kw) if dist else None
    env = make_env(n, hull_kw=dict(hull_model=hull_model, actuator_lag_s=lag), max_ep_len=L, auto_reset=True, seed=seed,
                   device=cuda_device)
    if dist:
        env.set_disturbance(**dist_kw)
    env.set_waves(**SEA)
    rng = np.random.default_rng(hull_model * 10 + int(lag > 0) + 100 * int(dist))
    eta0, nu0 = start_pose(rng, n)
    st = EO.new_state(spec, n)
    o_ref = WO.reset(spec, st, waves, dist=dO, eta=eta0, nu=nu0, seed=seed)
    o_gpu = env.reset(**init_kw(eta0, nu0))
    np.testing.assert_allclose(np_(o_gpu), o_ref, rtol=0, atol=5e-5)
    sig = waves.sigma[:, None]
    restarted_total = 0
    sg = env.get_state()
    for t in range(10):
        st['wave'] = np_(sg['wave']).astype(np.float64)
        st['wave_rate'] = np_(sg['wave_rate']).astype(np.float64)
        st['wave_omega'] = np_(sg['wave_omega']).astype(np.float64)
        if dist:
            st['current'], st['bias'] = np_(sg['current']).astype(np.float64), np_(sg['bias']).astype(np.float64)
        a = rng.uniform(-1.0, 1.0, (7, n)).astype(np.float32)
        o64, r64, d64, info = WO.step(spec, st, a.astype(np.float64), waves, dist=dO, seed=seed)
        o, r, d, inf = env.step(torch.as_tensor(a, device=cuda_device))
        sg = env.get_state()
        eta, nu = np_(sg['eta']).astype(np.float64), np_(sg['nu']).astype(np.float64)
        restarted = np_(inf['flags']) != 0
        keep = ~restarted
        assert ((np_(inf['flags']) & 1 != 0) == d64).all()
        np.testing.assert_allclose(eta[:, keep], st['eta'][:, keep], rtol=0, atol=2e-5)
        np.testing.assert_allclose(nu[:, keep], st['nu'][:, keep], rtol=0, atol=2e-6)
        np.testing.assert_allclose(np_(o)[:, keep], o64[:, keep], rtol=0, atol=5e-5)
        np.testing.assert_allclose(np_(r)[~d64 & keep], r64[~d64 & keep], rtol=0, atol=2e-4)
        w0 = st['wave_omega']
        assert (np.abs(np_(sg['wave'])[:, keep] - st['wave'][:, keep]) <= 2e-5 * sig).all()
        assert (np.abs(np_(sg['wave_rate'])[:, keep] - st['wave_rate'][:, keep]) <= 2e-5 * sig * w0[keep]).all()
        assert (np_(sg['wave_omega'])[keep] == w0[keep].astype(np.float32)).all()
        st['eta'][:, keep], st['nu'][:, keep] = eta[:, keep], nu[:, keep]
        if restarted.any():                                  # the kernel's restart: a new w0 and a stationary state
            WO.reset(spec, st, waves, dist=dO, mask=restarted, eta=eta, nu=nu, seed=seed)
            assert ulp_diff(np_(sg['wave_omega'])[restarted], st['wave_omega'][restarted]).max() <= 1
            w0 = st['wave_omega'][restarted]
            assert (np.abs(np_(sg['wave'])[:, restarted] - st['wave'][:, restarted]) <= 2e-6 * sig).all()
            assert (np.abs(np_(sg['wave_rate'])[:, restarted] - st['wave_rate'][:, restarted]) <= 2e-6 * sig * w0).all()
            o_re = WO.observe(spec, st)
            np.testing.assert_allclose(np_(o)[:, restarted], o_re[:, restarted], rtol=0, atol=5e-5)
            restarted_total += int(restarted.sum())
    assert restarted_total >= 2 * n                          # every env was cut at least twice (2-step episodes)


@pytest.mark.parametrize("how", ["reset", "reset_to", "restart"])
def test_draws_match_oracle(cuda_device, how):
    """w0 and the stationary state of the three kinds of reset come from the oracle's Philox blocks: w0 to 1 ulp, x and x'
    within fp32 tolerance."""
    n, seed = 10007, 31
    ids = np.arange(n)
    waves = WO.Waves(step_dt=DT, sigma=(0.2, 0.1, 0.05), peak_frequency=(0.5, 3.0), damping=0.3)
    env = make_env(n, seed=seed, auto_reset=True, max_ep_len=6, device=cuda_device, hull_kw=dict(frozen=True))
    env.set_waves(sigma=(0.2, 0.1, 0.05), peak_frequency=(0.5, 3.0), damping=0.3)
    word = np.zeros(n, dtype=np.int64)
    if how == "reset":
        env.reset(fraction=0.8)
    elif how == "reset_to":
        env.reset(**init_kw(np.zeros((3, n)), np.zeros((3, n))))
    else:
        env.reset()
        act = torch.zeros(7, n, device=cuda_device)
        act[4] = act[6] = 1.0
        episodes, prev_len = np.ones(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
        for _ in range(3):                                   # 3-step episodes: the third step cuts every env still running
            _, _, _, info = env.step(act)
            ended = np_(info['flags']) != 0
            word[ended] = (episodes[ended] << 16) | (prev_len[ended] + 1)
            episodes[ended] += 1
            prev_len = np_(env.get_state()['ep_len']).astype(np.int64)
        assert (episodes > 1).mean() > 0.99
        fresh = ended                                        # restarted by the last step: the state is the draw itself
    sg = env.get_state()
    w0, x, xd = waves.sample(seed, ids, word)
    sel = fresh if how == "restart" else np.ones(n, dtype=bool)
    assert sel.mean() > 0.5
    assert ulp_diff(np_(sg['wave_omega'])[sel], w0[sel]).max() <= 1
    sig = waves.sigma[:, None]
    assert (np.abs(np_(sg['wave'])[:, sel] - x[:, sel]) <= 2e-6 * sig).all()
    assert (np.abs(np_(sg['wave_rate'])[:, sel] - xd[:, sel]) <= 2e-6 * sig * w0[sel]).all()


def test_wave_statistics(cuda_device):
    """4 Mi envs on the null simulator: the std of x and of x' / w0 is within 1 % of sigma after the reset draw and after
    50 steps (stationarity); the lag-1 covariances E[s1 s0^T] match Phi P within 1 %; w0 is uniform (Kolmogorov-Smirnov)."""
    from scipy import stats
    n = 1 << 22
    sigma, lam = np.array([0.1, 0.2, 0.05]), 0.1
    env = make_env(n, seed=3, max_ep_len=10 ** 4, device=cuda_device, hull_kw=dict(frozen=True))
    env.set_waves(sigma=sigma, peak_frequency=(1.0, 2.0), damping=lam)
    env.reset()
    sg = env.get_state()
    w0 = np_(sg['wave_omega']).astype(np.float64)
    assert stats.kstest((w0[::16] - 1.0) / 1.0, 'uniform').pvalue > 1e-3
    act = torch.zeros(7, n, device=cuda_device)
    act[4] = act[6] = 1.0
    x0, v0 = np_(sg['wave']).astype(np.float64), np_(sg['wave_rate']).astype(np.float64)
    for x, v in ((x0, v0),):
        assert (np.abs(x.std(axis=1) / sigma - 1) < 0.01).all() and (np.abs((v / w0).std(axis=1) / sigma - 1) < 0.01).all()
    env.step(act)
    s1 = env.get_state()
    x1, v1 = np_(s1['wave']).astype(np.float64), np_(s1['wave_rate']).astype(np.float64)
    phi = WO.transition(w0, lam, DT)                             # E[s1 s0^T] = Phi P, P = sigma^2 diag(1, w0^2)
    s2 = sigma[:, None] ** 2
    for got, want in (((x1 * x0).mean(axis=1), (phi[0, 0] * s2).mean(axis=1)),
                      ((x1 * v0).mean(axis=1), (phi[0, 1] * w0 ** 2 * s2).mean(axis=1)),
                      ((v1 * x0).mean(axis=1), (phi[1, 0] * s2).mean(axis=1)),
                      ((v1 * v0).mean(axis=1), (phi[1, 1] * w0 ** 2 * s2).mean(axis=1))):
        assert (np.abs(got / want - 1) < 0.01).all(), (got, want)
    for _ in range(49):
        env.step(act)
    s50 = env.get_state()
    assert torch.equal(s50['wave_omega'], sg['wave_omega'])          # no restarts: w0 is the episode's
    x, v = np_(s50['wave']).astype(np.float64), np_(s50['wave_rate']).astype(np.float64)
    assert (np.abs(x.std(axis=1) / sigma - 1) < 0.01).all() and (np.abs((v / w0).std(axis=1) / sigma - 1) < 0.01).all()


def test_sharded_envs_equal_one_env(cuda_device):
    """Two envs holding the two halves of the batch (env_id_offset) step exactly like one env, with waves and the
    disturbance on."""
    n, h = 4000, 2000
    kw = dict(seed=8, auto_reset=True, max_ep_len=10, device=cuda_device)
    full, lo, hi = make_env(n, **kw), make_env(h, **kw), make_env(n - h, env_id_offset=h, **kw)
    for e in (full, lo, hi):
        e.set_disturbance(current_speed=(0.0, 0.2), current_direction=(0.0, TWO_PI), bias_std=(10.0, 10.0, 5.0),
                          bias_time_s=2.0)
        e.set_waves(**SEA)
        e.reset()
    g = torch.Generator(device=cuda_device)
    g.manual_seed(2)
    for t in range(12):
        a = torch.rand(7, n, device=cuda_device, generator=g) * 2 - 1
        o, r, _, _ = full.step(a)
        o1, r1, _, _ = lo.step(a[:, :h].contiguous())
        o2, r2, _, _ = hi.step(a[:, h:].contiguous())
        assert torch.equal(o, torch.cat([o1, o2], dim=1)) and torch.equal(r, torch.cat([r1, r2]))
    s, s1, s2 = full.get_state(), lo.get_state(), hi.get_state()
    for k in ("eta", "nu", "current", "bias", "wave", "wave_rate", "wave_omega", "ep_len"):
        assert torch.equal(s[k], torch.cat([s1[k], s2[k]], dim=-1)), k


def test_graph_rollout_equals_eager_and_draws_fresh_noise(cuda_device):
    """rollout(graph=True) with waves equals the eager rollout bitwise; two consecutive replays of one graph add different
    wave noise; a new set_waves between rollouts is not served by the graph captured with the old setting."""
    import ml4ca_b200 as M
    n, T, lam = 3000, 10, 0.1
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=cuda_device, seed=21)
    envs = [make_env(n, seed=9, auto_reset=True, max_ep_len=1000, device=cuda_device) for _ in range(2)]
    bufs = [M.TrajectoryBuffer(9, 7, T, n, device=cuda_device) for _ in range(2)]
    for e in envs:
        e.set_waves(**SEA)
        e.reset()

    def wave_state(e):
        s = e.get_state()
        return np_(s['wave']).astype(np.float64), np_(s['wave_rate']).astype(np.float64), np_(s['wave_omega']).astype(np.float64)
    prev, noise = wave_state(envs[1]), []
    for epoch in range(3):
        M.rollout(envs[0], ac, bufs[0], seed=5, start_step=epoch * T)
        M.rollout(envs[1], ac, bufs[1], seed=5, start_step=epoch * T, graph=True)
        for name in ("obs_buf", "act_buf", "rew_buf", "logp_buf", "done_buf"):
            assert torch.equal(getattr(bufs[0], name), getattr(bufs[1], name)), (epoch, name)
        sA, sB = envs[0].get_state(), envs[1].get_state()
        for k in ("eta", "nu", "prev_thrust", "ep_len", "wave", "wave_rate", "wave_omega"):
            assert torch.equal(sA[k], sB[k]), (epoch, k)
        cur = wave_state(envs[1])
        same = cur[2] == prev[2]                                  # no restart in this epoch: propagate the old state
        phi = WO.transition(prev[2], lam, DT)
        x, v = prev[0].copy(), prev[1].copy()
        for _ in range(T):
            x, v = phi[0, 0] * x + phi[0, 1] * v, phi[1, 0] * x + phi[1, 1] * v
        noise.append(np.where(same, cur[0] - x, np.nan))
        prev = cur
    assert all(e["graph"] is not None for e in bufs[1]._rollout_graphs.values())
    both = ~np.isnan(noise[1][0]) & ~np.isnan(noise[2][0])
    assert both.mean() > 0.5 and np.abs(noise[2] - noise[1])[:, both].max() > 0.05   # epochs 2 and 3: two replays of one graph
    for e in envs:
        e.set_waves(sigma=(0.02, 0.3, 0.1), peak_frequency=(2.0, 3.0), damping=0.5)
    for epoch in range(3, 5):
        M.rollout(envs[0], ac, bufs[0], seed=5, start_step=epoch * T)
        M.rollout(envs[1], ac, bufs[1], seed=5, start_step=epoch * T, graph=True)
        for name in ("obs_buf", "rew_buf", "done_buf"):
            assert torch.equal(getattr(bufs[0], name), getattr(bufs[1], name)), (epoch, name)
    assert len(bufs[1]._rollout_graphs) == 2


@pytest.mark.parametrize("n", [1001, 4096])
def test_step_host_equals_step(cuda_device, n):
    """ml4ca_env_step_host advances the wave rows chunk by chunk exactly like the device-buffer step."""
    kw = dict(seed=11, auto_reset=True, max_ep_len=12, device=cuda_device)
    A, B = make_env(n, **kw), make_env(n, **kw)
    for e in (A, B):
        e.set_waves(**SEA)
        e.reset()
    g = torch.Generator()
    g.manual_seed(n)
    h_obs, h_rew, h_done = torch.empty(9, n).pin_memory(), torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    for t in range(8):
        h_act = (torch.rand(7, n, generator=g) * 2.4 - 1.2).pin_memory()
        A.step_host(h_act, h_obs, h_rew, h_done)
        o, r, d, info = B.step(h_act.to(cuda_device))
        torch.cuda.synchronize()
        assert torch.equal(h_obs, o.cpu()) and torch.equal(h_rew, r.cpu()) and torch.equal(h_done, info['flags'].cpu())
    sA, sB = A.get_state(), B.get_state()
    for k in sA:
        assert torch.equal(sA[k], sB[k]), k


def test_cut_obs_and_observe_are_measured(cuda_device):
    """observe() returns the measured observation (after a reset: the reset's own observation, and after
    set_wave_state: the oracle's measured observation), and cut_obs holds the measured observation at the cut (what a
    twin without the restart returns there)."""
    from ml4ca_b200 import _lib
    n, L = 2048, 10
    spec = EO.EnvSpec('final', True, True, max_ep_len=L)
    A = make_env(n, seed=5, auto_reset=True, max_ep_len=L, device=cuda_device, hull_kw=dict(frozen=True))
    B = make_env(n, seed=5, auto_reset=False, max_ep_len=L, device=cuda_device, hull_kw=dict(frozen=True))
    for e in (A, B):
        e.set_waves(**SEA)
    o0 = A.reset()
    B.reset()
    assert torch.equal(A.observe(), o0)
    rng = np.random.default_rng(0)
    x, xd = rng.normal(size=(3, n)) * 0.05, rng.normal(size=(3, n)) * 0.05
    A.set_wave_state(motion=x, rate=xd)
    sg = A.get_state()
    st = {'eta': np_(sg['eta']).astype(np.float64), 'nu': np_(sg['nu']).astype(np.float64), 'ref': np.zeros((3, n)),
          'prev_thrust': np_(sg['prev_thrust']).astype(np.float64), 'wave': x.astype(np.float32).astype(np.float64),
          'wave_rate': xd.astype(np.float32).astype(np.float64)}
    np.testing.assert_allclose(np_(A.observe()), WO.observe(spec, st), rtol=0, atol=5e-5)
    em, nm = WO.measured(st['eta'], st['nu'], st['wave'], st['wave_rate'])
    np.testing.assert_allclose(np_(sg['eta_measured']), em, rtol=0, atol=2e-6)
    np.testing.assert_allclose(np_(sg['nu_measured']), nm, rtol=0, atol=1e-6)
    B.set_wave_state(motion=x, rate=xd)
    cut = torch.full((9, n), float('nan'), device=cuda_device)
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(A._handle, _lib.ptr(cut)), "ml4ca_env_set_cut_obs")
    act = torch.zeros(7, n, device=cuda_device)
    act[4] = act[6] = 1.0
    ok = torch.ones(n, dtype=torch.bool, device=cuda_device)
    T = A.max_ep_len                                                # the episode length in steps
    for t in range(T):
        oA, _, _, iA = A.step(act)
        oB, _, _, iB = B.step(act)
        ok &= iA['flags'] == iB['flags']
        if t < T - 1:
            ok &= iA['flags'] == 0
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(A._handle, None), "ml4ca_env_set_cut_obs")
    cut_envs = ok & (iA['flags'] == 2)
    assert float(cut_envs.float().mean()) > 0.5
    assert torch.equal(cut[:, cut_envs], oB[:, cut_envs])
    assert not torch.equal(oA[:, cut_envs], oB[:, cut_envs])       # the restart returned a new episode's observation


def test_state_access_and_bad_arguments(cuda_device):
    """set_wave_state / get_state round-trip, a set state holds (propagated) until that env's next reset; bad
    configurations and state access without waves raise ML4CA_ERR_INVALID with the library's message."""
    from ml4ca_b200 import _lib
    n = 64
    env = make_env(n, seed=2, device=cuda_device, hull_kw=dict(frozen=True))
    env.reset()
    assert "wave" not in env.get_state() and "eta_measured" not in env.get_state()
    for fn in ("ml4ca_env_set_wave_state", "ml4ca_env_get_waves"):
        assert getattr(_lib.lib(), fn)(env._handle, None, None, None, _lib.current_stream()) == ERR_INVALID
        assert "waves are not enabled" in _lib.lib().ml4ca_last_error().decode()
    with pytest.raises(_lib.Ml4caError, match="waves are not enabled"):
        env.set_wave_state(motion=torch.zeros(3, n, device=cuda_device))
    for bad, msg in ((dict(sigma=(0.1, -0.1, 0.0)), "sigma"), (dict(peak_frequency=(0.0, 1.0)), "peak frequency range"),
                     (dict(peak_frequency=(2.0, 1.0)), "peak frequency range"),
                     (dict(peak_frequency=(1.0, 16.0)), "omega_max \\* step_dt"), (dict(damping=0.0), "damping"),
                     (dict(damping=1.0), "damping"), (dict(sigma=(float('nan'), 0.0, 0.0)), "finite"),
                     (dict(peak_frequency=(1.0, float('inf'))), "finite")):
        kw = dict(SEA)
        kw.update(bad)
        with pytest.raises(_lib.Ml4caError, match=msg):
            env.set_waves(**kw)
        c = _lib.WaveCfg()
        for i, s in enumerate(kw['sigma']):
            c.sigma[i] = float(s)
        c.omega_min, c.omega_max = kw['peak_frequency']
        c.damping = kw['damping']
        assert _lib.lib().ml4ca_env_set_waves(env._handle, ctypes.byref(c), _lib.current_stream()) == ERR_INVALID
    env.set_waves(**SEA)
    s0 = env.get_state()
    w = torch.full((n,), 1.5, device=cuda_device)
    x, v = torch.randn(3, n, device=cuda_device) * 0.1, torch.randn(3, n, device=cuda_device) * 0.1
    env.set_wave_state(motion=x, rate=v, omega=w)
    st = env.get_state()
    assert torch.equal(st["wave"], x) and torch.equal(st["wave_rate"], v) and torch.equal(st["wave_omega"], w)
    assert torch.equal(st["eta"], s0["eta"]) and torch.equal(st["nu"], s0["nu"])
    act = torch.zeros(7, n, device=cuda_device)
    act[4] = act[6] = 1.0
    env.step(act)
    assert torch.equal(env.get_state()["wave_omega"], w)                      # w0 holds within the episode
    mask = torch.zeros(n, dtype=torch.bool)
    mask[::2] = True
    env.reset(mask=mask)
    st = env.get_state()
    m = mask.to(cuda_device)
    assert torch.equal(st["wave_omega"][~m], w[~m]) and not torch.equal(st["wave_omega"][m], w[m])
    assert ((st["wave_omega"] >= 1.0) & (st["wave_omega"] < 2.0)).all()
    env.set_waves(None)
    assert "wave" not in env.get_state()


def test_closed_loop_in_waves(cuda_device):
    """The PID + pseudoinverse allocator and the RL policy with the body-frame integrator run on the measured pose in
    waves; the metrics are finite and IAE scores the LF pose (the records are get_state()'s "eta")."""
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    n = 48
    mk = lambda: M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n,
                               device=cuda_device, max_ep_len=400)
    env = mk()
    env.set_waves(**SEA)
    rec = evaluate.run_allocator(env, method="pinv", max_ep_len=200)
    assert torch.isfinite(rec["metrics"]).all()
    assert torch.equal(rec["eta"][-1], env.get_state()["eta"])
    g = golden("policy_final_80x3.npz")
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=g["params"], device=cuda_device)
    env = mk()
    env.set_waves(**SEA)
    rec = evaluate.run_RL_policy(env, ac, max_ep_len=200, integrator=True)
    assert torch.isfinite(rec["metrics"]).all()


def test_ppo_graph_with_waves(cuda_device):
    """ppo(..., graph=True) for 3 epochs on an env with waves: finite statistics."""
    import ml4ca_b200 as M
    env = make_env(64, seed=3, auto_reset=True, device=cuda_device)
    env.set_waves(**SEA)
    ac, hist = M.ppo(env, steps_per_epoch=100, epochs=3, seed=1, graph=True)
    assert len(hist) == 3
    for h in hist:
        assert np.isfinite(h["LossPi"]) and np.isfinite(h["LossV"]) and np.isfinite(h["AverageStepReward"])
