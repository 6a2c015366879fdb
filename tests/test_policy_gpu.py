"""GPU parity of K4 (actor/critic MLP forward on tcgen05) and of the rollout loop built on it.

Tolerances: the tensor-core operands are fp16 (10-bit mantissa) with fp32 accumulation, so against the float64
oracle mu and v carry |err| <= 4e-3 * (1 + output range of the network) (measured ~1e-3); the sampled action
inherits the error of mu; logp_pi depends only on the noise and log_std and is checked at 1e-5.
"""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import mlp_oracle as MO

pytestmark = pytest.mark.gpu

CASES = [("glorot 64x64 leaky", dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2), "leaky_relu", None),
         ("glorot 64x64 tanh", dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2), "tanh", None),
         ("glorot 64x64 obs6 act5", dict(obs_dim=6, act_dim=5, hidden=64, n_hidden=2), "leaky_relu", None),
         ("shipped final 80x3", None, "leaky_relu", "policy_final_80x3.npz"),
         ("shipped limited 64x3", None, "leaky_relu", "policy_limited_64x3.npz"),
         # observation rows 12.. are loaded in place, not prefetched a tile ahead; with 15 inputs the constant-1 bias column is
         # the last K column of the first-layer operand
         ("glorot 64x3 obs13 act7", dict(obs_dim=13, act_dim=7, hidden=64, n_hidden=3), "leaky_relu", None),
         ("glorot 64x64 obs15 act1", dict(obs_dim=15, act_dim=1, hidden=64, n_hidden=2), "leaky_relu", None),
         ("glorot 80x3 tanh", dict(obs_dim=9, act_dim=7, hidden=80, n_hidden=3), "tanh", None)]

# Observation scales of the 9-state RevoltFinal input, then unit scales for wider inputs.
OBS_SCALE = [8, 8, .8, 1.4, .3, .5, 1, 1, 1.] + [1.] * 6


def load(dims, fixture):
    if fixture is None:
        return MO.glorot_params(dims, seed=3), dims
    g = golden(fixture)
    return g['params'], {k: int(g[k]) for k in ('obs_dim', 'act_dim', 'hidden', 'n_hidden')}


@pytest.mark.parametrize("name,dims,act,fixture", CASES)
# The persistent kernel works through the tiles in rounds of grid x G x 128 observations (148 SMs: 75 776 for the 64-wide nets,
# G = 4; 37 888 for the 80-wide ones, G = 2).  From the second round on, observation rows come from the one-tile-ahead prefetch
# and the mbarrier phase carries over.  75 777: 64-wide 2 rounds (the last with one live row), 80-wide 3 rounds; 228 328:
# 64-wide 4 rounds (the last tile holds 104 rows), 80-wide 7 rounds.
@pytest.mark.parametrize("n", [1, 127, 128 * 3 + 5, 70001, 75777, 228328])
def test_forward_matches_oracle(cuda_device, name, dims, act, fixture, n):
    import ml4ca_b200 as M
    flat, dims = load(dims, fixture)
    ac = M.ActorCritic(dims['obs_dim'], dims['act_dim'], (dims['hidden'],) * dims['n_hidden'], act, params=flat,
                       device=cuda_device, seed=11)
    g = torch.Generator(device=cuda_device); g.manual_seed(n)
    scale = torch.tensor(OBS_SCALE, device=cuda_device)[:dims['obs_dim'], None]
    obs = (torch.rand(dims['obs_dim'], n, device=cuda_device, generator=g) * 2 - 1) * scale
    pi, v, logp, mu = ac.step(obs, deterministic=True, return_mu=True)
    ref = MO.forward(flat, dims, obs.cpu().numpy().astype(np.float64), act)
    # error scale = the output range of the network on this input distribution (the value head of the shipped
    # nets spans ~ +-300 with heavy cancellation: a single small output still carries the absolute fp16 error)
    rng = np.random.default_rng(0)
    probe = MO.forward(flat, dims, rng.uniform(-1, 1, (dims['obs_dim'], 4096)) * scale.cpu().numpy(), act)
    tol_mu = 4e-3 * (1 + np.abs(probe['mu']).max())
    tol_v = 4e-3 * (1 + np.abs(probe['v']).max())
    np.testing.assert_allclose(mu.cpu().numpy().reshape(dims['act_dim'], n), ref['mu'], rtol=0, atol=tol_mu)
    np.testing.assert_allclose(v.cpu().numpy().reshape(n), ref['v'], rtol=0, atol=tol_v)
    np.testing.assert_array_equal(pi.cpu().numpy(), mu.cpu().numpy())          # deterministic action = mu
    # log-likelihood of mu under the policy: sum -0.5 (2 log_std + log 2 pi)  (core.py:42-46)
    want = float((-0.5 * (2 * ref['log_std'] + np.log(2 * np.pi))).sum())
    np.testing.assert_allclose(logp.cpu().numpy().reshape(n), want, rtol=0, atol=1e-5)


def test_sampling_and_loglikelihood(cuda_device):
    """pi = mu + eps * exp(log_std) with eps ~ N(0, 1) (core.py:85); logp_pi consistent with the sample."""
    import ml4ca_b200 as M
    dims = dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2)
    flat = MO.glorot_params(dims, seed=3)
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", params=flat, device=cuda_device, seed=5)
    n = 1 << 18
    obs = torch.rand(9, n, device=cuda_device) * 2 - 1
    pi, v, logp, mu = ac.step(obs, step=3, return_mu=True)
    pi2, _, _, _ = ac.step(obs, step=3, return_mu=True)
    pi3, _, _, _ = ac.step(obs, step=4, return_mu=True)
    assert torch.equal(pi, pi2) and not torch.equal(pi, pi3)         # counter RNG: reproducible per (seed, env, step)
    log_std = MO.unflatten(flat, dims)[1]
    eps = ((pi - mu).cpu().numpy().astype(np.float64)) / np.exp(log_std)[:, None]
    assert abs(eps.mean()) < 5e-3 and abs(eps.std() - 1.0) < 5e-3
    assert abs(np.mean(eps ** 3)) < 2e-2 and abs(np.mean(eps ** 4) - 3.0) < 5e-2
    assert abs(np.corrcoef(eps[0], eps[1])[0, 1]) < 5e-3 and abs(np.corrcoef(eps[0, :-1], eps[0, 1:])[0, 1]) < 5e-3
    want = MO.gaussian_likelihood(pi.cpu().numpy().T.astype(np.float64), mu.cpu().numpy().T.astype(np.float64), log_std)
    np.testing.assert_allclose(logp.cpu().numpy(), want, rtol=0, atol=2e-4)
    # a shard starting at global id 1000 draws the same noise as envs 1000.. of the full batch
    pis, _, _ = ac.step(obs[:, 1000:3000].contiguous(), step=3, env_id_offset=1000)
    assert torch.equal(pis, pi[:, 1000:3000])


@pytest.mark.parametrize("act_dim", [7, 3])
def test_exploration_noise_matches_philox_oracle(cuda_device, act_dim):
    """eps = (pi - mu) / exp(log_std) draw for draw against oracle/philox.py::policy_normals: key (seed_lo, seed_hi ^ 0xAC710A)
    with a non-zero upper seed word, two Philox blocks per (env, step) (eps[4..7] from the second), global env ids that cross
    into the id's high word (shard offset 2^32 - 1000).

    Error model, per draw.  Box-Muller in the kernel: r = sqrtf(-2 __logf(u)), (c, s) = __sincosf(2 pi f).  __logf carries
    an absolute error <= 2^-21.41 for u in [0.5, 1] and <= 3 ulp below, so r^2 is off by dr2 = 2 max(2^-21.41, 3 2^-23 |ln u|)
    and r by min(sqrt(dr2), dr2 / r): loose where u -> 1 and r -> 0.  The angle: 2 pi rounded to fp32 and the fp32 product
    (<= 2^-21 together) plus the absolute error of sin.approx / cos.approx over [0, 2 pi) (2^-20.5) give r 2^-19.8.
    Recovering eps from the fp32 outputs adds half an ulp of pi over exp(log_std), and expf (2 ulp), sqrtf and the product
    r c in fp32 add |eps| 2^-21.  Measured on a B200: largest error 3.4e-5 (act_dim 7) and 4.1e-6 (act_dim 3), both at
    r < 0.01 (1.0e-4 over 2^20 envs); nowhere more than 0.36 of the bound."""
    import ml4ca_b200 as M
    from oracle import philox as PH
    dims = dict(obs_dim=9, act_dim=act_dim, hidden=64, n_hidden=2)
    flat = MO.glorot_params(dims, seed=3)
    seed = 0xC0FFEE1234ABCDEF
    ac = M.ActorCritic(9, act_dim, (64, 64), "leaky_relu", params=flat, device=cuda_device, seed=seed)
    n, off, step = 1 << 16, (1 << 32) - 1000, 0x80000011
    obs = torch.rand(9, n, device=cuda_device, generator=torch.Generator(device=cuda_device).manual_seed(2)) * 2 - 1
    pi, _, _, mu = ac.step(obs, step=step, env_id_offset=off, return_mu=True)
    pi, mu = pi.cpu().numpy().astype(np.float64), mu.cpu().numpy().astype(np.float64)
    sd = np.exp(MO.unflatten(flat, dims)[1])[:, None]
    eps = (pi - mu) / sd
    ids = np.arange(n, dtype=np.uint64) + np.uint64(off)
    want = PH.policy_normals(seed, ids, step)[:act_dim]
    # the uniforms of each Box-Muller pair, for the error model
    k1 = ((seed >> 32) ^ 0xAC710A) & 0xFFFFFFFF
    u = []
    for block in (0, 1):
        q = PH.philox4x32(ids & np.uint64(0xFFFFFFFF), ids >> np.uint64(32), np.full(n, step, np.uint64),
                          np.full(n, block, np.uint64), seed & 0xFFFFFFFF, k1)
        u += [PH.unit_open(q[0]).astype(np.float64)] * 2 + [PH.unit_open(q[2]).astype(np.float64)] * 2
    u = np.stack(u)[:act_dim]
    r = np.sqrt(-2.0 * np.log(u))
    dr2 = 2.0 * np.maximum(2.0 ** -21.41, 3 * 2.0 ** -23 * np.abs(np.log(u)))
    tol = (np.minimum(np.sqrt(dr2), dr2 / np.maximum(r, 1e-30)) + r * 2.0 ** -19.8
           + 0.5 * np.spacing(np.abs(pi).astype(np.float32)).astype(np.float64) / sd + np.abs(want) * 2.0 ** -21)
    assert np.isfinite(eps).all()
    err = np.abs(eps - want)
    assert (err <= tol).all(), (err.max(), (err / tol).max(), np.unravel_index(np.argmax(err / tol), err.shape))
    # two blocks, not one: eps[4..7] are not a copy of eps[0..3]
    if act_dim == 7:
        assert np.abs(eps[4:7] - eps[0:3]).max() > 1.0
    # the noise follows the global id: the same rows at offset 0 draw other noise
    pi0, _, _ = ac.step(obs, step=step, env_id_offset=0)
    assert not torch.equal(pi0.cpu(), torch.as_tensor(pi.astype(np.float32)))


def test_parameter_update_roundtrip(cuda_device):
    import ml4ca_b200 as M
    dims = dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2)
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", params=MO.glorot_params(dims, seed=3), device=cuda_device)
    obs = torch.rand(9, 1000, device=cuda_device)
    _, v0, _ = ac.step(obs, deterministic=True)
    new = MO.glorot_params(dims, seed=4)
    ac.parameters().copy_(torch.as_tensor(new, device=cuda_device))
    ac.refresh()
    _, v1, _ = ac.step(obs, deterministic=True)
    ref = MO.forward(new, dims, obs.cpu().numpy().astype(np.float64), "leaky_relu")
    assert not torch.allclose(v0, v1)
    np.testing.assert_allclose(v1.cpu().numpy(), ref['v'], rtol=0, atol=4e-3 * (1 + np.abs(ref['v']).max()))


def test_unsupported_shapes_fail_loudly(cuda_device):
    import ml4ca_b200 as M
    from ml4ca_b200._lib import Ml4caError
    with pytest.raises(Ml4caError):
        M.ActorCritic(9, 7, (32, 32), device=cuda_device)
    with pytest.raises(AssertionError):
        M.ActorCritic(9, 7, (64, 80), device=cuda_device)


@pytest.mark.parametrize("reset_acts", [False, True])
def test_rollout_matches_stepwise_reference_semantics(cuda_device, reset_acts):
    """T steps of rollout() == the reference loop `a = pi(o); o, r, d = env.step(a)` (ppo.py:290-302) driven
    step by step through the separate policy / env kernels, including the stale-thrust tail of the observation
    the agent acts on and in-kernel restarts of finished episodes."""
    import ml4ca_b200 as M
    from ml4ca_b200.env import RevoltFinal, StandInHull
    dims = dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2)
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", params=MO.glorot_params(dims, seed=3), device=cuda_device, seed=21)
    n, T = 20000, 12
    mk = lambda: RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=cuda_device, seed=9,
                             auto_reset=True, max_ep_len=16, reset_acts=reset_acts)   # 16 * 10 / 20 = 8-step episodes
    envA, envB = mk(), mk()
    o = envA.reset()
    envB.reset()
    buf = M.TrajectoryBuffer(9, 7, T, n, device=cuda_device)
    M.rollout(envB, ac, buf, seed=21, start_step=100)
    ended = 0
    for t in range(T):
        pi, v, logp = ac.step(o, step=100 + t)
        assert torch.equal(buf.obs_buf[t], o)
        assert torch.equal(buf.act_buf[t], pi) and torch.equal(buf.val_buf[t], v) and torch.equal(buf.logp_buf[t], logp)
        o, r, d, info = envA.step(pi)
        np.testing.assert_allclose(buf.rew_buf[t].cpu().numpy(), r.cpu().numpy(), rtol=0, atol=2e-6)
        assert torch.equal(buf.done_buf[t], info['flags'])
        ended += int((info['flags'] != 0).sum())
    assert ended >= n          # every env restarted at least once (8-step episodes, 12 steps)
    sA, sB = envA.get_state(), envB.get_state()
    for k in ('eta', 'nu', 'prev_thrust', 'angles'):
        np.testing.assert_allclose(sB[k].cpu().numpy(), sA[k].cpu().numpy(), rtol=0, atol=2e-6)
    assert torch.equal(sA['ep_len'], sB['ep_len'])


def test_graph_rollout_equals_eager_rollout(cuda_device):
    """rollout(graph=True): the T steps captured into a CUDA graph and replayed with the Philox step number taken from a
    device counter reproduce the eager launches bit for bit, epoch after epoch (first call eager, second captures)."""
    import ml4ca_b200 as M
    from ml4ca_b200.env import RevoltFinal, StandInHull
    dims = dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2)
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", params=MO.glorot_params(dims, seed=3), device=cuda_device, seed=21)
    n, T = 3000, 10
    mk = lambda: RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=cuda_device, seed=9,
                             auto_reset=True, max_ep_len=16)
    envA, envB = mk(), mk()
    envA.reset(); envB.reset()
    bufA = M.TrajectoryBuffer(9, 7, T, n, device=cuda_device)
    bufB = M.TrajectoryBuffer(9, 7, T, n, device=cuda_device)
    for epoch, start in enumerate([0, T, 2 * T, (1 << 32) - 4]):       # the last one wraps the 32-bit step number
        M.rollout(envA, ac, bufA, seed=5, start_step=start)
        M.rollout(envB, ac, bufB, seed=5, start_step=start, graph=True)
        for name in ("obs_buf", "act_buf", "rew_buf", "logp_buf", "done_buf"):
            assert torch.equal(getattr(bufA, name), getattr(bufB, name)), (epoch, name)
        assert torch.equal(bufA.val_buf[:T], bufB.val_buf[:T])
        sA, sB = envA.get_state(), envB.get_state()
        for k in ("eta", "nu", "prev_thrust", "angles", "ep_len"):
            assert torch.equal(sA[k], sB[k]), (epoch, k)
    assert bufB._rollout_graphs and all(e["graph"] is not None for e in bufB._rollout_graphs.values())
    # eager calls after a capture are unaffected by the counter
    a1 = ac.step(bufA.obs_buf[0], step=7)[0]
    a2 = ac.step(bufA.obs_buf[0], step=7)[0]
    assert torch.equal(a1, a2)
