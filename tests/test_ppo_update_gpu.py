"""GPU parity of K6 (PPO gradients, loss statistics, Adam) against the float64 restatement of ppo.py:234-250, which is
itself cross-checked against torch autograd in tests/test_ppo_cpu.py."""
import numpy as np
import pytest
import torch

from oracle import mlp_oracle as MO
from oracle import ppo_oracle as PO

pytestmark = pytest.mark.gpu

DIMS = dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2)


def _batch(T, n, seed):
    rng = np.random.default_rng(seed)
    obs = rng.normal(size=(T, 9, n)).astype(np.float32) * np.array([2, 2, .3, .5, .1, .2, .5, .5, .5], dtype=np.float32)[None, :, None]
    act = rng.normal(size=(T, 7, n)).astype(np.float32)
    adv = rng.normal(size=(T, n)).astype(np.float32)
    ret = (rng.normal(size=(T, n)) * 3).astype(np.float32)
    return obs, act, adv, ret


def _flatten(x):          # [T, c, n] -> [T * n, c] in (t, i) order
    return np.ascontiguousarray(np.moveaxis(x, 1, 2).reshape(-1, x.shape[1])).astype(np.float64)


@pytest.fixture(params=["tensor_core", "fp32"])
def precision(request, lib_built):
    """Both gradient kernels: tcgen05 (fp16 operands, default) and the fp32 CUDA-core one."""
    from ml4ca_b200 import _lib
    prev = _lib.lib().ml4ca_ppo_use_fp32(1 if request.param == "fp32" else 0)
    yield request.param
    _lib.lib().ml4ca_ppo_use_fp32(prev)


@pytest.mark.parametrize("activation", ["leaky_relu", "tanh"])
@pytest.mark.parametrize("T,n", [(1, 128), (3, 1000), (2, 40000)])
def test_gradients_and_statistics(cuda_device, precision, activation, T, n):
    import ml4ca_b200 as M
    # stated tolerances of the two kernels.  Tensor cores: fp16 operands give ~1e-3; on top of that a pre-activation
    # within fp16 rounding of zero can take the other leaky-ReLU branch, a per-sample effect that averages out as 1/sqrt(N)
    gtol, stol = (2e-4, 1e-5) if precision == "fp32" else (3e-3 + 0.5 / np.sqrt(T * n), 3e-2)
    if precision == "tensor_core" and activation == "tanh":
        gtol += 1.2e-2        # tanh.approx.f16x2 (MUFU, 2^-11) in the forward pass biases logp by ~1 %; every shipped model is leaky-ReLU
    flat = MO.glorot_params(DIMS, seed=5)
    flat = (flat + np.random.default_rng(1).normal(size=flat.size).astype(np.float32) * 0.05).astype(np.float32)   # non-zero biases
    ac = M.ActorCritic(9, 7, (64, 64), activation, params=flat, device=cuda_device)
    obs, act, adv, ret = _batch(T, n, seed=T * n)
    # logp_old from a slightly different policy, so that ratios spread around 1 and some samples clip
    fo = MO.forward((flat * 1.02).astype(np.float32), DIMS, _flatten(obs).T, activation)
    logp_old = MO.gaussian_likelihood(_flatten(act), fo["mu"].T, fo["log_std"]).astype(np.float32).reshape(T, n)
    g64, info = PO.ppo_gradients(flat.astype(np.float64), DIMS, _flatten(obs), _flatten(act), adv.reshape(-1).astype(np.float64),
                                 ret.reshape(-1).astype(np.float64), logp_old.reshape(-1).astype(np.float64), 0.2, activation)
    upd = M.PPOUpdater(ac)
    dev = lambda x: torch.as_tensor(x, device=cuda_device).contiguous()
    data = (dev(obs), dev(act), dev(adv), dev(ret), dev(logp_old))
    n_pi = ac.var_counts[0]
    N = float(T * n)
    s, c = upd._grad(0, data, T, n)
    assert c == N
    g_pi = upd.flat[:ac.num_params].cpu().numpy().astype(np.float64) / N
    assert (g_pi[n_pi:] == 0).all()                     # the v block is untouched by the pi pass
    scale = np.abs(g64[:n_pi]).max()
    np.testing.assert_allclose(g_pi[:n_pi], g64[:n_pi], rtol=0, atol=gtol * scale)
    assert abs(-s[0] / N - info["pi_loss"]) < stol * max(1, abs(info["pi_loss"]))
    assert abs(s[2] / N - info["approx_kl"]) < stol * max(1e-3, info["approx_kl"]) + 1e-7 + (0 if precision == "fp32" else 1e-3)
    assert abs(s[3] / N - info["approx_ent"]) < stol * abs(info["approx_ent"])
    assert abs(s[4] / N - info["clipfrac"]) <= 2.0 / N + (1e-4 if precision == "fp32" else 1e-2)   # ratios within rounding of the clip edge may flip
    s, c = upd._grad(1, data, T, n)
    g_v = upd.flat[:ac.num_params].cpu().numpy().astype(np.float64) / N
    assert (g_v[:n_pi] == 0).all()
    scale = np.abs(g64[n_pi:]).max()
    np.testing.assert_allclose(g_v[n_pi:], g64[n_pi:], rtol=0, atol=gtol * scale)
    assert abs(s[1] / N - info["v_loss"]) < stol * info["v_loss"]


@pytest.mark.parametrize("hidden", [(80, 80, 80), (64, 64, 64)])
@pytest.mark.parametrize("activation", ["leaky_relu", "tanh"])
def test_gradients_of_the_reference_network_shapes(cuda_device, precision, hidden, activation):
    """The reference trains 80 x 80 x 80 by default (train.py:30-32; every shipped checkpoint is 80^3 or 64^3): those shapes
    run on the tensor-core gradient kernel as well (csrc/ppo_update_tc.cu, templated on width and depth; default) and on the
    generic fp32 kernel (csrc/ppo_update_generic.cu; ml4ca_ppo_use_fp32).  Same float64 restatement, the stated tolerance of each
    kernel; batch sizes around the reference's own (4 x 400 samples) and one ragged multi-tile case."""
    import ml4ca_b200 as M
    dims = dict(obs_dim=9, act_dim=7, hidden=hidden[0], n_hidden=len(hidden))
    flat = MO.glorot_params(dims, seed=11)
    flat = (flat + np.random.default_rng(2).normal(size=flat.size).astype(np.float32) * 0.05).astype(np.float32)
    ac = M.ActorCritic(9, 7, hidden, activation, params=flat, device=cuda_device)
    # (80^3 has two tensor-core variants, picked by the batch size: one tile group with two threads per row up to two waves of
    # tiles, two groups on shared weight-gradient accumulators beyond -- the 80 000-sample case; 296 / 297 tiles sit on either side
    # of the switch, 446 tiles is an odd count: the second group of some CTAs gets one tile less)
    deep = ((2, 40000), (1, 296 * 128), (1, 297 * 128 - 5), (1, 445 * 128 + 1)) if hidden == (80, 80, 80) and activation == "leaky_relu" else ()
    for T, n in ((4, 400), (3, 1037)) + deep:
        # tensor cores: the fp16 rounding of the operands enters once per layer, so the 3e-3 of the two-layer config scales with the depth
        gtol, stol = (2e-4, 1e-5) if precision == "fp32" else (3e-3 * len(hidden) / 2.0 + 0.5 / np.sqrt(T * n), 3e-2)
        if precision == "tensor_core" and activation == "tanh":
            gtol += 1.2e-2        # tanh.approx.f16x2 in the forward pass (see test_gradients_and_statistics)
        tc = precision != "fp32"
        obs, act, adv, ret = _batch(T, n, seed=T * n + 1)
        fo = MO.forward((flat * 1.02).astype(np.float32), dims, _flatten(obs).T, activation)
        logp_old = MO.gaussian_likelihood(_flatten(act), fo["mu"].T, fo["log_std"]).astype(np.float32).reshape(T, n)
        g64, info = PO.ppo_gradients(flat.astype(np.float64), dims, _flatten(obs), _flatten(act), adv.reshape(-1).astype(np.float64),
                                     ret.reshape(-1).astype(np.float64), logp_old.reshape(-1).astype(np.float64), 0.2, activation)
        upd = M.PPOUpdater(ac)
        dev = lambda x: torch.as_tensor(x, device=cuda_device).contiguous()
        data = (dev(obs), dev(act), dev(adv), dev(ret), dev(logp_old))
        n_pi, N = ac.var_counts[0], float(T * n)
        s, c = upd._grad(0, data, T, n)
        assert c == N
        g_pi = upd.flat[:ac.num_params].cpu().numpy().astype(np.float64) / N
        assert (g_pi[n_pi:] == 0).all()
        np.testing.assert_allclose(g_pi[:n_pi], g64[:n_pi], rtol=0, atol=gtol * np.abs(g64[:n_pi]).max())
        assert abs(-s[0] / N - info["pi_loss"]) < stol * max(1, abs(info["pi_loss"]))
        assert abs(s[2] / N - info["approx_kl"]) < stol * max(1e-3, info["approx_kl"]) + 1e-7 + (1e-3 if tc else 0)
        assert abs(s[3] / N - info["approx_ent"]) < stol * abs(info["approx_ent"])
        assert abs(s[4] / N - info["clipfrac"]) <= 2.0 / N + (1e-2 if tc else 1e-4)
        s, c = upd._grad(1, data, T, n)
        g_v = upd.flat[:ac.num_params].cpu().numpy().astype(np.float64) / N
        assert (g_v[:n_pi] == 0).all()
        np.testing.assert_allclose(g_v[n_pi:], g64[n_pi:], rtol=0, atol=gtol * np.abs(g64[n_pi:]).max())
        assert abs(s[1] / N - info["v_loss"]) < stol * info["v_loss"]


def test_ppo_trains_the_shipped_architecture(cuda_device):
    """ppo() end to end with the reference's default network (80 x 80 x 80, leaky-ReLU) at the reference's batch size
    (4 envs x 400 steps, config.json): the update runs, stops on KL, and the value loss falls within an epoch."""
    import ml4ca_b200 as M
    from ml4ca_b200.env import RevoltFinal, StandInHull
    env = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=4, device=cuda_device, seed=3, auto_reset=True)
    ac, hist = M.ppo(env, steps_per_epoch=400, epochs=2, seed=3, hidden_sizes=(80, 80, 80), activation="leaky_relu")
    assert ac.hidden_sizes == (80, 80, 80)
    for h in hist:
        assert np.isfinite(h["LossPi"]) and np.isfinite(h["LossV"]) and np.isfinite(h["KL"])
        assert h["DeltaLossV"] < 0 and 0 <= h["StopIter"] < 80
    assert hist[-1]["TotalEnvInteracts"] == 2 * 400 * 4


@pytest.mark.parametrize("target_kl,want_stop", [(1e-9, 1), (1.0, 11)])
@pytest.mark.parametrize("hidden", [(64, 64), (80, 80, 80)])
def test_graph_update_equals_eager_update(cuda_device, hidden, target_kl, want_stop):
    """PPOUpdater.update(graph=True): the pi / v iterations, the device-side KL stop (ppo.py:268-271) and the closing loss
    passes replayed from ONE CUDA graph leave the parameters, the Adam moments and the logger's numbers where the
    host-driven loop leaves them -- same stopping iterations, over several epochs (the step counts of the bias correction
    carry over)."""
    import ml4ca_b200 as M
    T, n = 4, 4096
    obs, act, adv, ret = _batch(T, n, seed=17)
    res = []
    for use_graph in (False, True, False):
        ac = M.ActorCritic(9, 7, hidden, "leaky_relu", device=cuda_device, seed=4)
        buf = M.TrajectoryBuffer(9, 7, T, n, device=cuda_device)
        # target 1e-9: approx-KL is 0 before the first step (logp_old is the current policy's) and > 0 after it, so the loop stops
        # at iteration 1 whatever the rounding; target 1: it never stops
        upd = M.PPOUpdater(ac, train_pi_iters=12, train_v_iters=9, target_kl=target_kl)
        infos = []
        for epoch in range(3):
            buf.obs_buf.copy_(torch.as_tensor(obs)); buf.act_buf.copy_(torch.as_tensor(act))
            buf.adv_buf.copy_(torch.as_tensor(adv) * (1.0 + 0.1 * epoch)); buf.ret_buf.copy_(torch.as_tensor(ret))
            with torch.no_grad():
                _, _, logp = ac.step(buf.obs_buf.permute(1, 0, 2).reshape(9, -1).contiguous(), deterministic=True)
            # log-likelihood of the stored actions under the current policy = logp_old (ratio starts at 1)
            fo = MO.forward(ac.parameters().cpu().numpy(), dict(obs_dim=9, act_dim=7, hidden=hidden[0], n_hidden=len(hidden)),
                            _flatten(obs).T, "leaky_relu")
            lp = MO.gaussian_likelihood(_flatten(act), fo["mu"].T, fo["log_std"]).astype(np.float32).reshape(T, n)
            buf.logp_buf.copy_(torch.as_tensor(lp))
            infos.append(upd.update(buf, graph=use_graph))
        res.append((ac.parameters().clone(), upd.m1.clone(), upd.m2.clone(), infos, upd.t_pi, upd.t_v))
    (pa, m1a, m2a, ia, tpa, tva), (pb, m1b, m2b, ib, tpb, tvb), (pc, _, _, ic, _, _) = res
    assert [i["StopIter"] for i in ia] == [i["StopIter"] for i in ib]
    # (the tensor-core forward differs from the float64 logp_old by ~1e-3, which already exceeds 1.5e-9 at iteration 0)
    assert all(i["StopIter"] <= want_stop for i in ia) if want_stop == 1 else all(i["StopIter"] == want_stop for i in ia)
    assert (tpa, tva) == (tpb, tvb)
    # Not bit-equal: the gradient kernels sum per-CTA partials with atomicAdd, so two runs of EITHER path differ in the last
    # bits of the gradient, and Adam turns a gradient component at noise level into a step of +-lr whatever its size
    # (profiles/ppo_graph_noise_r2.txt: eager vs eager ends 2e-3..7e-3 of the travelled distance apart, graph vs eager the same).
    # The graph must therefore land as close to the host-driven loop as a second host-driven run does.
    ac0 = M.ActorCritic(9, 7, hidden, "leaky_relu", device=cuda_device, seed=4)
    p0 = ac0.parameters().clone()
    moved = float((pa - p0).norm())
    floor = float((pa - pc).norm()) / moved
    dist = float((pa - pb).norm()) / moved
    assert floor < 0.05 and dist < 0.05, (floor, dist)
    # the noise level itself scatters between pairs of runs (80^3 on the tensor-core kernel, second part of that record: eager vs
    # eager 6.3e-3 .. 1.9e-2, graph vs graph 5.4e-3 .. 1.7e-2, eager vs graph 6.3e-3 .. 1.9e-2), so one measured floor is no sharp
    # bound for another pair: three floors or the largest recorded level, whichever is larger
    # (the iteration counts themselves are compared exactly above: StopIter and the Adam step counts)
    assert dist <= max(3.0 * floor, 3e-2), (floor, dist)
    for a, b in zip(ia, ib):
        for k in ("LossPi", "LossV", "KL", "Entropy", "ClipFrac", "DeltaLossPi", "DeltaLossV"):
            assert abs(a[k] - b[k]) <= 2e-3 * max(1.0, abs(a[k])), (k, a[k], b[k])


def test_adam_step_matches_tf1_formula(cuda_device):
    from ml4ca_b200 import _lib
    rng = np.random.default_rng(0)
    m = 5001
    p = rng.normal(size=m).astype(np.float32); g = rng.normal(size=m).astype(np.float32) * 123.0
    p64, m1, m2 = p.astype(np.float64), np.zeros(m), np.zeros(m)
    tp, tg = torch.as_tensor(p, device=cuda_device), torch.as_tensor(g, device=cuda_device)
    t1, t2 = torch.zeros(m, device=cuda_device), torch.zeros(m, device=cuda_device)
    for t in range(1, 6):
        _lib.check(_lib.lib().ml4ca_adam_step(m, _lib.ptr(tp), _lib.ptr(tg), _lib.ptr(t1), _lib.ptr(t2), 3e-4, 0.9, 0.999, 1e-8, t,
                                              1.0 / 123.0, _lib.current_stream()))
        p64, m1, m2 = PO.adam_step(p64, g.astype(np.float64) / 123.0, m1, m2, 3e-4, t)
    np.testing.assert_allclose(tp.cpu().numpy(), p64, rtol=0, atol=2e-6)


def test_update_improves_the_surrogate_and_stops_on_kl(cuda_device):
    """PPOUpdater.update on a synthetic buffer: the v-loss falls, the pi iterations stop once approx-KL > 1.5 target,
    and the parameters actually used by the tensor-core forward follow the fp32 master copy (refresh)."""
    import ml4ca_b200 as M
    T, n = 4, 8192
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=cuda_device, seed=1)
    obs, act, adv, ret = _batch(T, n, seed=9)
    buf = M.TrajectoryBuffer(9, 7, T, n, device=cuda_device)
    buf.obs_buf.copy_(torch.as_tensor(obs)); buf.act_buf.copy_(torch.as_tensor(act))
    buf.adv_buf.copy_(torch.as_tensor(adv)); buf.ret_buf.copy_(torch.as_tensor(ret))
    flat0 = ac.parameters().clone()
    fo = MO.forward(flat0.cpu().numpy(), DIMS, _flatten(obs).T, "leaky_relu")
    buf.logp_buf.copy_(torch.as_tensor(MO.gaussian_likelihood(_flatten(act), fo["mu"].T, fo["log_std"]).reshape(T, n), dtype=torch.float32))
    mu_before = ac.step(buf.obs_buf[0], deterministic=True)[0].clone()
    upd = M.PPOUpdater(ac, train_pi_iters=80, train_v_iters=20, target_kl=1e-4)
    info = upd.update(buf)
    assert info["DeltaLossV"] < 0 and info["DeltaLossPi"] < 0
    assert 0 < info["StopIter"] < 79 and info["KL"] > 1.5e-4      # stopped by the KL rule, with that step applied
    assert not torch.equal(flat0, ac.parameters())
    assert not torch.equal(mu_before, ac.step(buf.obs_buf[0], deterministic=True)[0])


def test_training_run_writes_the_reference_log_format(cuda_device, tmp_path):
    """ppo() with logger_kwargs: progress.txt carries exactly the columns of the reference's shipped runs
    (tests/golden/progress_header.txt = first line of data/finalmodel/finconttothighbowder_s0/progress.txt), one row per
    epoch, and the episode statistics agree with a NumPy scan of the recorded buffer."""
    import json, os
    import ml4ca_b200 as M
    from conftest import GOLDEN
    n, T = 4096, 60
    env = M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=cuda_device, seed=3,
                        auto_reset=True, max_ep_len=40)                       # 20-step episodes
    seen = []
    ac, hist = M.ppo(env, steps_per_epoch=T, epochs=2, train_pi_iters=3, train_v_iters=3, seed=3,
                     logger_kwargs=dict(output_dir=str(tmp_path), exp_name="t"), logger=seen.append)
    lines = open(os.path.join(tmp_path, "progress.txt")).read().splitlines()
    assert lines[0] == open(os.path.join(GOLDEN, "progress_header.txt")).read().strip()
    assert len(lines) == 3 and len(lines[1].split("\t")) == len(lines[0].split("\t"))
    row = dict(zip(lines[0].split("\t"), map(float, lines[2].split("\t"))))
    assert row["Epoch"] == 1 and row["TotalEnvInteracts"] == 2 * T * n and row["EpLen"] <= 20 + 1e-9
    assert row["MinEpRet"] <= row["AverageEpRet"] <= row["MaxEpRet"] and row["StdVVals"] >= 0
    cfg = json.load(open(os.path.join(tmp_path, "config.json")))
    assert cfg["gamma"] == 0.99 and cfg["ac_kwargs"]["hidden_sizes"] == [64, 64]
    assert hist[-1]["Episodes"] >= 2 * n          # 60 steps of <= 20-step episodes: at least two ended per env per epoch


def test_episode_statistics_kernel(cuda_device):
    import torch
    from ml4ca_b200 import _lib
    rng = np.random.default_rng(0)
    n, T = 777, 50
    rew = rng.normal(size=(2, T, n)).astype(np.float32)
    done = (rng.random((2, T, n)) < 0.07).astype(np.uint8) * rng.integers(1, 4, (2, T, n)).astype(np.uint8)
    run_ret, run_len = torch.zeros(n, device=cuda_device), torch.zeros(n, dtype=torch.int32, device=cuda_device)
    s5 = torch.zeros(2, 5, dtype=torch.float64, device=cuda_device)
    acc, ln = np.zeros(n), np.zeros(n, dtype=np.int64)
    for e in range(2):                             # two consecutive buffers: episodes carry over the boundary
        r_t, d_t = torch.as_tensor(rew[e], device=cuda_device), torch.as_tensor(done[e], device=cuda_device)
        _lib.check(_lib.lib().ml4ca_episode_stats(n, T, _lib.ptr(r_t), _lib.ptr(d_t), _lib.ptr(run_ret), _lib.ptr(run_len),
                                                  _lib.ptr(s5[0]), _lib.ptr(s5[1]), _lib.current_stream()))
        rets, lens = [], []
        for t in range(T):
            acc += rew[e, t]; ln += 1
            end = done[e, t] != 0
            rets += list(acc[end]); lens += list(ln[end])
            acc[end] = 0; ln[end] = 0
        got = s5.cpu().numpy()
        want_r = [np.sum(rets), np.sum(np.square(rets)), len(rets), np.min(rets), np.max(rets)]
        want_l = [np.sum(lens), np.sum(np.square(lens)), len(lens), np.min(lens), np.max(lens)]
        np.testing.assert_allclose(got[0], want_r, rtol=2e-5, atol=1e-4)
        np.testing.assert_allclose(got[1], want_l, rtol=1e-12)
    x = torch.as_tensor(rew[0], device=cuda_device)
    _lib.check(_lib.lib().ml4ca_stats5(x.numel(), _lib.ptr(x), _lib.ptr(s5[0]), _lib.current_stream()))
    np.testing.assert_allclose(s5[0].cpu().numpy(), [rew[0].astype(np.float64).sum(), (rew[0].astype(np.float64) ** 2).sum(), rew[0].size,
                                                     rew[0].min(), rew[0].max()], rtol=1e-9)


def test_ppo_learns_station_keeping_at_the_reference_batch_size(cuda_device):
    """End-to-end learning check at the reference's own batch size (4 envs x 400 steps = 1600 interactions per epoch,
    config.json): the reference's shipped run (data/finalmodel/finconttothighbowder_s0/progress.txt) starts at
    AverageEpRet -21 / AverageVVals -0.7 and passes AverageEpRet 787 / VVals 231 at 638 k interactions; the GPU pipeline
    (rollout, GAE, tensor-core update) on the stand-in hull starts at the same level and is well past +1 reward per step
    after 200 epochs = 320 k interactions (measured over several runs: 1.2-2.3 per step, EpRet 500-800, VVals 175-260).  Loose thresholds: fp32
    atomics make the run non-reproducible at the last bit."""
    import ml4ca_b200 as M
    from ml4ca_b200.env import RevoltFinal, StandInHull
    env = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=4, device=cuda_device, seed=0, auto_reset=True)
    ac, hist = M.ppo(env, steps_per_epoch=400, epochs=200, seed=0)
    first, last = hist[0], hist[-10:]
    assert -0.6 < first["AverageStepReward"] < 0.1 and abs(first["AverageVVals"]) < 5
    assert np.mean([h["AverageStepReward"] for h in last]) > 0.5       # runs differ (atomics): 1.2 - 2.3 observed
    assert np.mean([h["AverageVVals"] for h in last]) > 50
    assert np.mean([h["EpLen"] for h in last if h["Episodes"] > 0]) > 200



@pytest.mark.parametrize("hidden", [(64, 64), (64, 64, 64), (80, 80, 80)])
@pytest.mark.parametrize("obs_dim,act_dim", [(9, 5), (6, 3), (9, 6)])
def test_gradients_for_the_other_env_classes(cuda_device, precision, hidden, obs_dim, act_dim):
    """RevoltLimited (5 actions; the shipped 64^3 model), RevoltSimple (3 actions, 6 observations), RevoltFinal without continuous
    angles (6 actions): the gradient kernels with run-time observation / action dims (the 9 -> 7 case is a compile-time
    specialisation), every network shape, both precisions, against the float64 restatement."""
    import ml4ca_b200 as M
    T, n = 2, 20000
    dims = dict(obs_dim=obs_dim, act_dim=act_dim, hidden=hidden[0], n_hidden=len(hidden))
    flat = MO.glorot_params(dims, seed=17)
    flat = (flat + np.random.default_rng(5).normal(size=flat.size).astype(np.float32) * 0.05).astype(np.float32)
    ac = M.ActorCritic(obs_dim, act_dim, hidden, "leaky_relu", params=flat, device=cuda_device)
    obs, act, adv, ret = _batch(T, n, seed=obs_dim * 10 + act_dim)
    obs, act = np.ascontiguousarray(obs[:, :obs_dim]), np.ascontiguousarray(act[:, :act_dim])
    fo = MO.forward((flat * 1.02).astype(np.float32), dims, _flatten(obs).T, "leaky_relu")
    logp_old = MO.gaussian_likelihood(_flatten(act), fo["mu"].T, fo["log_std"]).astype(np.float32).reshape(T, n)
    g64, info = PO.ppo_gradients(flat.astype(np.float64), dims, _flatten(obs), _flatten(act), adv.reshape(-1).astype(np.float64),
                                 ret.reshape(-1).astype(np.float64), logp_old.reshape(-1).astype(np.float64), 0.2, "leaky_relu")
    # fp32 kernels: 2e-4 of the largest component as everywhere.  Tensor cores: 40 000 samples keep the 1 / sqrt(N) term of the bound
    # (leaky-ReLU branch flips within fp16 rounding of zero) below the rounding term; for these input / output shapes two or three
    # components of ~10^4 reach 1.6 x the rounding term of the 9 -> 7 tests (measured), so it is stated 2 x larger here
    upd = M.PPOUpdater(ac)
    dev = lambda x: torch.as_tensor(x, device=cuda_device).contiguous()
    data = (dev(obs), dev(act), dev(adv), dev(ret), dev(logp_old))
    n_pi, N = ac.var_counts[0], float(T * n)

    def close(g, ref):
        gtol = 2e-4 if precision == "fp32" else 2.0 * 3e-3 * len(hidden) / 2.0 + 0.5 / np.sqrt(T * n)
        np.testing.assert_allclose(g, ref, rtol=0, atol=gtol * np.abs(ref).max())
    s, c = upd._grad(0, data, T, n)
    g_pi = upd.flat[:ac.num_params].cpu().numpy().astype(np.float64) / N
    assert c == N and (g_pi[n_pi:] == 0).all()
    close(g_pi[:n_pi], g64[:n_pi])
    s, c = upd._grad(1, data, T, n)
    g_v = upd.flat[:ac.num_params].cpu().numpy().astype(np.float64) / N
    assert (g_v[:n_pi] == 0).all()
    close(g_v[n_pi:], g64[n_pi:])
