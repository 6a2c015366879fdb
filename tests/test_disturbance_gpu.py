"""GPU checks of the environmental disturbance (ml4ca_env_set_disturbance): the DIST variant of the env-step kernel, its
Philox draws and its Python surface, against the float64 restatement (tests/disturbance_oracle.py).

Tolerances are those of tests/test_env_gpu.py: observation <= 5e-5, reward <= 2e-4, hull state 2e-5 (position) /
2e-6 (velocity); the bias force <= 1e-6 relative to its scale."""
import numpy as np
import pytest
import torch

import disturbance_oracle as DO
from conftest import golden
from oracle import env_oracle as EO

pytestmark = pytest.mark.gpu

TWO_PI = 2 * np.pi


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
    eta = rng.uniform(-1, 1, (3, n)) * np.array([[5.0], [5.0], [0.5]])
    nu = rng.uniform(-1, 1, (3, n)) * np.array([[0.8], [0.15], [0.3]])
    return eta.astype(np.float32).astype(np.float64), nu.astype(np.float32).astype(np.float64)


def np_(t):
    return t.cpu().numpy()


@pytest.mark.parametrize("kind,cont,ext,lag,exact", [('limited', False, False, None, True), ('limited', False, True, 0.92, False),
                                                     ('final', True, True, None, False), ('final', True, True, 0.92, False)])
def test_zero_disturbance_equals_calm_water(cuda_device, kind, cont, ext, lag, exact):
    """The DIST kernel with zero ranges returns what the default dispatch returns: obs, reward, flags and state over 500 steps
    with episode-length cuts, terminations and in-kernel restarts (n odd: both run one env per thread).  The two kernels are
    compiled separately, and outside the correctly rounded (_rn) operations the compiler is free to form multiply-adds
    differently in each, so bit-for-bit equality is asserted only where it holds on the B200 build (RevoltLimited without the
    lag); elsewhere the comparison is at fp32 level on the envs whose flags have agreed so far."""
    n, act_dim = 4099, (7 if cont else 5)
    hull_kw = None if lag is None else dict(hull_model=1, actuator_lag_s=lag)
    kw = dict(seed=4, auto_reset=True, max_ep_len=60, reset_acts=True, device=cuda_device)
    A, B = make_env(n, kind, cont, ext, hull_kw, **kw), make_env(n, kind, cont, ext, hull_kw, **kw)
    B.set_disturbance(current_speed=(0.0, 0.0), current_direction=(0.0, 0.0), bias_std=(0.0, 0.0, 0.0), bias_time_s=3.0)
    A.reset(), B.reset()
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
        else:
            sync &= iA['flags'] == iB['flags']
            assert float((oA - oB)[:, sync].abs().max()) <= 1e-4 and float((rA - rB)[sync].abs().max()) <= 5e-4, t
        if t % 50 == 49:
            sA, sB = A.get_state(), B.get_state()
            for k in ("eta", "nu", "prev_thrust", "angles", "ep_len"):
                assert torch.equal(sA[k], sB[k]) if exact else float((sA[k] - sB[k])[..., sync].abs().max()) <= 1e-3, (t, k)
            assert (sB["current"] == 0).all() and (sB["bias"] == 0).all()
    assert restarts > n and float(sync.float().mean()) > 0.99


@pytest.mark.parametrize("hull_model,lag", [(0, 0.0), (0, 0.5), (1, 0.0), (1, 0.92)])
def test_disturbed_step_matches_oracle(cuda_device, hull_model, lag):
    """One step at a time against the float64 oracle with current and a slowly varying bias on, through episode-length
    cuts and in-kernel restarts (which draw a new current and bias)."""
    n, seed = 2053, 12
    dist_kw = dict(current_speed=(0.0, 0.2), current_direction=(-np.pi, np.pi), bias_std=(15.0, 10.0, 8.0), bias_time_s=4.0)
    spec = EO.EnvSpec('final', True, True, max_ep_len=12, hull_model=hull_model, actuator_lag_s=lag)
    dist = DO.Disturbance(step_dt=float(np.float32(0.2)), **dist_kw)
    env = make_env(n, hull_kw=dict(hull_model=hull_model, actuator_lag_s=lag), max_ep_len=12, auto_reset=True, seed=seed,
                   device=cuda_device)
    env.set_disturbance(**dist_kw)
    rng = np.random.default_rng(hull_model * 10 + int(lag > 0))
    eta0, nu0 = start_pose(rng, n)
    st = EO.new_state(spec, n)
    DO.reset(spec, st, dist, eta=eta0, nu=nu0, seed=seed)
    env.reset(**init_kw(eta0, nu0))
    sg = env.get_state()
    np.testing.assert_allclose(np_(sg['current']), st['current'], rtol=0, atol=1e-7)
    np.testing.assert_allclose(np_(sg['bias']), st['bias'], rtol=0, atol=2e-6 * 15)
    scale = np.array([15.0, 10.0, 8.0])[:, None]
    restarted_total = 0
    for t in range(10):
        st['current'], st['bias'] = np_(sg['current']).astype(np.float64), np_(sg['bias']).astype(np.float64)
        a = rng.uniform(-1.0, 1.0, (7, n)).astype(np.float32)
        o64, r64, d64, info = DO.step(spec, st, a.astype(np.float64), dist, seed=seed)
        o, r, d, inf = env.step(torch.as_tensor(a, device=cuda_device))
        sg = env.get_state()
        eta, nu = np_(sg['eta']).astype(np.float64), np_(sg['nu']).astype(np.float64)
        restarted = np_(inf['flags']) != 0
        keep = ~restarted
        assert restarted.mean() < 0.2 or info['truncated'].all()
        np.testing.assert_allclose(eta[:, keep], st['eta'][:, keep], rtol=0, atol=2e-5)
        np.testing.assert_allclose(nu[:, keep], st['nu'][:, keep], rtol=0, atol=2e-6)
        np.testing.assert_allclose(np_(o)[:, keep], o64[:, keep], rtol=0, atol=5e-5)
        np.testing.assert_allclose(np_(r)[~d64 & keep], r64[~d64 & keep], rtol=0, atol=2e-4)
        assert (np.abs(np_(sg['bias'])[:, keep] - st['bias'][:, keep]) <= 1e-6 * scale).all()
        st['eta'][:, keep], st['nu'][:, keep] = eta[:, keep], nu[:, keep]
        if restarted.any():                                  # the kernel's restart: a new current and bias
            DO.reset(spec, st, dist, mask=restarted, eta=eta, nu=nu, seed=seed)
            np.testing.assert_allclose(np_(sg['current'])[:, restarted], st['current'][:, restarted], rtol=0, atol=1e-7)
            assert (np.abs(np_(sg['bias'])[:, restarted] - st['bias'][:, restarted]) <= 2e-6 * scale).all()
            restarted_total += int(restarted.sum())
    assert restarted_total >= n                              # every env was cut at least once (6-step episodes)


@pytest.mark.parametrize("how", ["reset", "reset_to", "restart"])
def test_draws_match_oracle(cuda_device, how):
    """Current and bias draws of the three kinds of reset come from the oracle's Philox blocks: the speed bits exactly
    (direction range (0, 0) makes the stored current V itself), direction and normals within fp32 tolerance."""
    n, seed = 10007, 31
    ids = np.arange(n)
    for dist_kw in (dict(current_speed=(0.0, 0.25), current_direction=(0.0, 0.0), bias_std=(1.0, 2.0, 4.0)),
                    dict(current_speed=(1.0, 1.0), current_direction=(-np.pi, np.pi))):
        env = make_env(n, seed=seed, auto_reset=True, max_ep_len=6, device=cuda_device, hull_kw=dict(frozen=True))
        env.set_disturbance(**dist_kw)
        dist = DO.Disturbance(**dist_kw)
        if how == "reset":
            env.reset(fraction=0.8)
            word = np.zeros(n, dtype=np.int64)
        elif how == "reset_to":
            env.reset(**init_kw(np.zeros((3, n)), np.zeros((3, n))))
            word = np.zeros(n, dtype=np.int64)
        else:
            env.reset()
            act = torch.zeros(7, n, device=cuda_device)
            act[4] = act[6] = 1.0
            word = np.zeros(n, dtype=np.int64)               # the episode word of each env's last reset
            episodes, prev_len = np.ones(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
            for _ in range(3):                               # 3-step episodes: the third step cuts every env still running
                _, _, _, info = env.step(act)
                ended = np_(info['flags']) != 0
                word[ended] = (episodes[ended] << 16) | (prev_len[ended] + 1)
                episodes[ended] += 1
                prev_len = np_(env.get_state()['ep_len']).astype(np.int64)
            assert (episodes > 1).mean() > 0.99
        sg = env.get_state()
        cur, bias = np_(sg['current']), np_(sg['bias'])
        cur64, bias64 = dist.sample(seed, ids, word)
        if dist_kw['current_direction'] == (0.0, 0.0):
            u = DO.current_units(seed, ids, word)[0]
            np.testing.assert_array_equal(cur[0], (0.25 * u).astype(np.float32))
            assert (cur[1] == 0).all()
            np.testing.assert_allclose(bias, bias64, rtol=0, atol=2e-6 * 4)
        else:
            beta = np.arctan2(cur[1], cur[0])
            beta64 = np.arctan2(cur64[1], cur64[0])
            assert np.abs(np.angle(np.exp(1j * (beta - beta64)))).max() < 1e-6
            np.testing.assert_allclose(np.hypot(cur[0], cur[1]), 1.0, rtol=0, atol=1e-6)
            assert (bias == 0).all()


def test_disturbance_statistics(cuda_device):
    """4 Mi envs: speed and direction are uniform on their ranges (Kolmogorov-Smirnov); the bias keeps its std and has
    lag-1 autocorrelation a = exp(-step_dt / T_b) (both within 1 %)."""
    from scipy import stats
    n = 1 << 22
    env = make_env(n, seed=3, max_ep_len=10 ** 4, device=cuda_device, hull_kw=dict(frozen=True))
    sigma, T_b = np.array([20.0, 10.0, 5.0]), 2.0
    env.set_disturbance(current_speed=(0.05, 0.2), current_direction=(-1.0, 2.0), bias_std=sigma, bias_time_s=T_b)
    env.reset()
    sg = env.get_state()
    cur = np_(sg['current']).astype(np.float64)
    V, beta = np.hypot(cur[0], cur[1]), np.arctan2(cur[1], cur[0])
    sub = slice(0, n, 16)
    assert stats.kstest((V[sub] - 0.05) / 0.15, 'uniform').pvalue > 1e-3
    assert stats.kstest((beta[sub] + 1.0) / 3.0, 'uniform').pvalue > 1e-3
    b0 = np_(sg['bias']).astype(np.float64)
    act = torch.zeros(7, n, device=cuda_device)
    act[4] = act[6] = 1.0
    env.step(act)
    b1 = np_(env.get_state()['bias']).astype(np.float64)
    a = np.exp(-float(np.float32(0.2)) / T_b)
    for b in (b0, b1):
        assert (np.abs(b.std(axis=1) / sigma - 1) < 0.01).all()
    corr = (b0 * b1).mean(axis=1) / (b0.std(axis=1) * b1.std(axis=1))
    assert (np.abs(corr / a - 1) < 0.01).all(), corr


def test_sharded_envs_equal_one_env(cuda_device):
    """Two envs holding the two halves of the batch (env_id_offset) step exactly like one env."""
    n, h = 4000, 2000
    kw = dict(seed=8, auto_reset=True, max_ep_len=10, device=cuda_device)
    dist_kw = dict(current_speed=(0.0, 0.2), current_direction=(0.0, TWO_PI), bias_std=(10.0, 10.0, 5.0), bias_time_s=2.0)
    full, lo, hi = make_env(n, **kw), make_env(h, **kw), make_env(n - h, env_id_offset=h, **kw)
    for e in (full, lo, hi):
        e.set_disturbance(**dist_kw)
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
    for k in ("eta", "nu", "current", "bias", "ep_len"):
        assert torch.equal(s[k], torch.cat([s1[k], s2[k]], dim=-1)), k


def test_graph_rollout_equals_eager_and_draws_fresh_noise(cuda_device):
    """rollout(graph=True) on a disturbed env equals the eager rollout bitwise; two consecutive replays add different
    bias noise (the per-step stream is keyed by the episode word, which moves on)."""
    import ml4ca_b200 as M
    n, T = 3000, 10
    dist_kw = dict(current_speed=(0.0, 0.1), current_direction=(0.0, TWO_PI), bias_std=(10.0, 10.0, 5.0), bias_time_s=2.0)
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=cuda_device, seed=21)
    envs = [make_env(n, seed=9, auto_reset=True, max_ep_len=1000, device=cuda_device) for _ in range(2)]
    bufs = [M.TrajectoryBuffer(9, 7, T, n, device=cuda_device) for _ in range(2)]
    for e in envs:
        e.set_disturbance(**dist_kw)
        e.reset()
    a = np.exp(-float(np.float32(0.2)) / 2.0)
    bias, noise = [np_(envs[1].get_state()['bias'])], []
    for epoch in range(3):
        M.rollout(envs[0], ac, bufs[0], seed=5, start_step=epoch * T)
        M.rollout(envs[1], ac, bufs[1], seed=5, start_step=epoch * T, graph=True)
        for name in ("obs_buf", "act_buf", "rew_buf", "logp_buf", "done_buf"):
            assert torch.equal(getattr(bufs[0], name), getattr(bufs[1], name)), (epoch, name)
        sA, sB = envs[0].get_state(), envs[1].get_state()
        for k in ("eta", "nu", "prev_thrust", "ep_len", "current", "bias"):
            assert torch.equal(sA[k], sB[k]), (epoch, k)
        bias.append(np_(sB['bias']))
        noise.append(bias[-1] - a ** T * bias[-2])
    assert all(e["graph"] is not None for e in bufs[1]._rollout_graphs.values())
    assert np.abs(noise[2] - noise[1]).max() > 1.0                # epochs 2 and 3 are two replays of one graph


@pytest.mark.parametrize("n", [1001, 4096])
def test_step_host_equals_step(cuda_device, n):
    """ml4ca_env_step_host advances the disturbance rows chunk by chunk exactly like the device-buffer step."""
    kw = dict(seed=11, auto_reset=True, max_ep_len=12, device=cuda_device)
    dist_kw = dict(current_speed=(0.0, 0.2), current_direction=(0.0, TWO_PI), bias_std=(10.0, 10.0, 5.0), bias_time_s=2.0)
    A, B = make_env(n, **kw), make_env(n, **kw)
    for e in (A, B):
        e.set_disturbance(**dist_kw)
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


def test_state_access_and_bad_arguments(cuda_device):
    """set_disturbance_state / get_state round-trip; a set state holds until that env's next reset; bad arguments raise
    with the library's message; get_state has no disturbance keys in calm water."""
    from ml4ca_b200 import _lib
    n = 64
    env = make_env(n, seed=2, device=cuda_device, hull_kw=dict(frozen=True))
    env.reset()
    assert "current" not in env.get_state()
    with pytest.raises(_lib.Ml4caError, match="no disturbance is enabled"):
        env.set_disturbance_state(current=torch.zeros(2, n, device=cuda_device))
    for bad, msg in ((dict(current_speed=(-0.1, 0.1)), "current speed range"), (dict(current_speed=(0.2, 0.1)), "current speed range"),
                     (dict(current_direction=(1.0, 0.0)), "direction range"), (dict(bias_std=(1.0, -1.0, 0.0)), "bias_std"),
                     (dict(bias_time_s=-1.0), "bias_time_s"), (dict(current_speed=(0.0, float('nan'))), "finite")):
        with pytest.raises(_lib.Ml4caError, match=msg):
            env.set_disturbance(**bad)
    env.set_disturbance(current_speed=(0.0, 0.2), bias_std=(5.0, 5.0, 2.0), bias_time_s=0.0)
    cur = torch.rand(2, n, device=cuda_device) * 0.1
    bias = torch.randn(3, n, device=cuda_device)
    env.set_disturbance_state(current=cur, bias=bias)
    act = torch.zeros(7, n, device=cuda_device)
    act[4] = act[6] = 1.0
    for _ in range(3):
        env.step(act)
    st = env.get_state()
    assert torch.equal(st["current"], cur) and torch.equal(st["bias"], bias)    # T_b = 0: constant over the episode
    mask = torch.zeros(n, dtype=torch.bool)
    mask[::2] = True
    env.reset(mask=mask)
    st = env.get_state()
    m = mask.to(cuda_device)
    assert torch.equal(st["current"][:, ~m], cur[:, ~m]) and torch.equal(st["bias"][:, ~m], bias[:, ~m])
    assert not torch.equal(st["current"][:, m], cur[:, m]) and not torch.equal(st["bias"][:, m], bias[:, m])
    env.set_disturbance(None)
    assert "current" not in env.get_state()


def test_closed_loop_under_current(cuda_device):
    """Integral action at work: the PID + pseudoinverse allocator holds station within 0.5 m after 120 s in a 0.1 m/s
    current from every fixed test pose; the RL policy with the deployment node's body-frame integrator runs and its
    integrator state becomes non-zero (its offset is recorded in profiles/disturbance_r3.md, not asserted)."""
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    n = 48
    mk = lambda: M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n,
                               device=cuda_device, max_ep_len=1200)
    env = mk()
    env.set_disturbance(current_speed=(0.1, 0.1), current_direction=(0.0, TWO_PI))
    rec = evaluate.run_allocator(env, method="pinv", max_ep_len=600)
    eta = np_(rec["eta"])
    d1 = np.hypot(eta[-1, 0], eta[-1, 1])
    assert (d1 < 0.5).all(), d1
    g = golden("policy_final_80x3.npz")
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=g["params"], device=cuda_device)
    env = mk()
    env.set_disturbance(current_speed=(0.1, 0.1), current_direction=(0.0, TWO_PI))
    rec = evaluate.run_RL_policy(env, ac, max_ep_len=300, integrator=True)
    assert torch.isfinite(rec["metrics"]).all()
    assert (rec["integrator"].abs().sum(dim=0) > 0).any()


def test_ppo_graph_on_a_disturbed_env(cuda_device):
    """ppo(..., graph=True) for 3 epochs on a disturbed env: finite statistics."""
    import ml4ca_b200 as M
    env = make_env(64, seed=3, auto_reset=True, device=cuda_device)
    env.set_disturbance(current_speed=(0.0, 0.1), current_direction=(0.0, TWO_PI), bias_std=(5.0, 5.0, 2.0), bias_time_s=10.0)
    ac, hist = M.ppo(env, steps_per_epoch=100, epochs=3, seed=1, graph=True)
    assert len(hist) == 3
    for h in hist:
        assert np.isfinite(h["LossPi"]) and np.isfinite(h["LossV"]) and np.isfinite(h["AverageStepReward"])
