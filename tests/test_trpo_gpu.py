"""GPU parity of the TRPO / NPG pieces (ml4ca_trpo_policy_mu, ml4ca_trpo_kl_grad, TRPOUpdater, trpo()) against the
float64 restatement of spinup/algos/tf1/trpo (oracle/trpo_oracle.py).

Every network shape (64 x 64, 64^3, 80^3), the run-time observation / action dims of the other env classes, both gradient
kernels.  Tolerances: mu 2e-5 (1 + max|mu|) (fp32 kernels vs float64; 2e-5 absolute at 64 x 64, 9 -> 7); surrogate / KL
gradients 2e-4 of the largest component; the Hessian-vector product (central difference of the KL gradient vs exact double
back-propagation) 3e-3 of its norm; a whole policy update: same accepted line-search index, step direction cosine > 0.999,
parameters within 2 % of the step length.  The tensor-core kernel: see _check_mu_and_kl_gradient."""
import numpy as np
import pytest
import torch

from oracle import mlp_oracle as MO
from oracle import trpo_oracle as TO

pytestmark = pytest.mark.gpu

DIMS = dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2)
OBS_SCALE = np.array([2, 2, .3, .5, .1, .2, .5, .5, .5])


def _flatten(x):          # [T, c, n] -> [T * n, c] in (t, i) order
    return np.ascontiguousarray(np.moveaxis(x, 1, 2).reshape(-1, x.shape[1])).astype(np.float64)


def _setup(cuda_device, T, n, activation="leaky_relu", seed=0, dims=DIMS):
    """A buffer sampled from the policy itself (actions = mu + eps sigma, logp_old = its likelihood), normalised
    advantages correlated with the first action so that the surrogate has a clear descent direction."""
    import ml4ca_b200 as M
    O, A = dims["obs_dim"], dims["act_dim"]
    rng = np.random.default_rng(seed)
    flat = MO.glorot_params(dims, seed=5)
    flat = (flat + rng.normal(size=flat.size).astype(np.float32) * 0.05).astype(np.float32)
    ac = M.ActorCritic(O, A, (dims["hidden"],) * dims["n_hidden"], activation, params=flat, device=cuda_device)
    obs = (rng.normal(size=(T, O, n)) * OBS_SCALE[None, :O, None]).astype(np.float32)
    npi = TO.n_pi(dims)
    theta = flat[:npi].astype(np.float64)
    ls = theta[-A:]
    prob0 = TO.Problem(dims, activation, _flatten(obs), np.zeros((T * n, A)), np.zeros(T * n), np.zeros(T * n),
                       np.zeros((T * n, A)), ls)
    mu64 = prob0.mu(theta)                                         # [N, A]
    eps = rng.normal(size=mu64.shape)
    act64 = mu64 + eps * np.exp(ls)
    logp = MO.gaussian_likelihood(act64, mu64, ls)
    adv = eps[:, 0] + 0.5 * rng.normal(size=T * n)
    adv = (adv - adv.mean()) / adv.std()
    ret = rng.normal(size=T * n) * 3
    unflat = lambda a, c: np.ascontiguousarray(np.moveaxis(a.reshape(T, n, c), 2, 1)).astype(np.float32)
    dev = lambda x: torch.as_tensor(np.ascontiguousarray(x), device=cuda_device)
    act32 = unflat(act64, A)
    data = [dev(obs), dev(act32), dev(adv.reshape(T, n).astype(np.float32)), dev(ret.reshape(T, n).astype(np.float32)),
            dev(logp.reshape(T, n).astype(np.float32))]
    prob = TO.Problem(dims, activation, _flatten(obs), _flatten(act32), adv.astype(np.float32), logp.astype(np.float32),
                      mu64, ls)
    return ac, data, prob, theta, mu64


def _policy_mu(ac, data, T, n, tensor_core):
    """ml4ca_trpo_policy_mu on the selected kernel -> [T, act, n] (pre-filled with 7.0: rows it fails to write show)."""
    from ml4ca_b200 import _lib
    L = _lib.lib()
    mu = torch.full((T, ac.act_dim, n), 7.0, device=data[0].device)
    prev = L.ml4ca_trpo_use_tensor_cores(1 if tensor_core else 0)
    try:
        _lib.check(L.ml4ca_trpo_policy_mu(ac._handle, n, T, _lib.ptr(data[0]), _lib.ptr(mu), _lib.current_stream()))
    finally:
        L.ml4ca_trpo_use_tensor_cores(prev)
    return mu


def _check_mu_and_kl_gradient(cuda_device, dims, kernel, activation, T, n, mu_atol=None):
    """The means, d_kl and its gradient at theta_old and at a perturbed theta (log_std moved as well), and the surrogate
    gradient, against float64.  Tolerances: fp32 kernels 2e-5 (1 + max|mu|) on the means, 2e-4 of the largest gradient
    component.  Tensor cores: fp16 operands, 4e-3 (1 + max|mu|) on the means with two hidden layers and 6e-3 with three; the
    gradient bound of the PPO tests (3e-3 per two layers, twice that for the run-time dims, + 0.5 / sqrt(N) for leaky-ReLU
    branch flips).  d_kl against float64: its first-order sensitivity to that error on the means; against the kernel's own
    means (recomputed in float64 from them): 1e-4 relative, as on the fp32 kernels."""
    import ml4ca_b200 as M
    tc = kernel == "tensor_core"
    O, A, NL = dims["obs_dim"], dims["act_dim"], dims["n_hidden"]
    N = T * n
    ac, data, prob, theta, mu64 = _setup(cuda_device, T, n, activation, dims=dims)
    mu_scale = 1 + np.abs(mu64).max()
    if mu_atol is None:
        mu_atol = (2e-5 if not tc else 4e-3 if NL == 2 else 6e-3) * mu_scale
    buf_mu = _policy_mu(ac, data, T, n, tc)
    np.testing.assert_allclose(_flatten(buf_mu.cpu().numpy()), mu64, rtol=0, atol=mu_atol)
    upd = M.TRPOUpdater(ac, kernel=kernel)
    upd._mu_tc = buf_mu                                                # mu_old of the tensor-core passes: its own means
    ls_old = torch.as_tensor(theta[-A:].astype(np.float32), device=cuda_device)
    full = data + [ls_old, buf_mu]
    g0, kl0 = upd._kl(full, T, n, tensor_core=tc)
    assert abs(kl0) < 1e-6 and np.abs(g0).max() < 1e-5                # d_kl and its gradient vanish at theta_old
    # away from theta_old, log_std included
    rng = np.random.default_rng(3)
    th1 = theta + rng.normal(size=theta.size) * 0.01
    th1[-A:] += 0.02
    upd._set_pi(th1)
    g1, kl1 = upd._kl(full, T, n, tensor_core=tc)
    mu_old = _flatten(buf_mu.cpu().numpy())
    prob.mu_old = torch.as_tensor(mu_old)                              # the kernel's own means, like the product path
    th1_32 = th1.astype(np.float32).astype(np.float64)
    g64, kl64 = prob.kl_gradient(th1_32)
    ls1, ls0 = th1_32[-A:], theta[-A:].astype(np.float32).astype(np.float64)
    var_old = np.exp(2 * ls0) + TO.EPS

    def kl_of(mu1):
        return float(np.mean(np.sum(0.5 * (((mu1 - mu_old) ** 2 + np.exp(2 * ls1)) / var_old - 1) + ls0 - ls1, axis=1)))
    mu1_k = _flatten(_policy_mu(ac, data, T, n, tc).cpu().numpy())    # the means the KL pass sees at th1
    assert abs(kl1 - kl_of(mu1_k)) < 1e-4 * kl64 + 1e-7
    if tc:
        d = np.abs(prob.mu(th1_32) - mu_old)
        assert abs(kl1 - kl64) < float(np.mean(np.sum((d * mu_atol + 0.5 * mu_atol ** 2) / var_old, axis=1))) + 1e-7
        gtol = 3e-3 * NL / 2.0 * (1 if (O, A) == (9, 7) else 2) + 0.5 / np.sqrt(N)
    else:
        assert abs(kl1 - kl64) < 1e-4 * kl64 + 1e-7
        gtol = 2e-4
    np.testing.assert_allclose(g1, g64, rtol=0, atol=gtol * np.abs(g64).max())
    # the surrogate gradient at theta_old (ratio = 1 up to fp32 rounding of logp; the fp32 kernel in both modes)
    upd._set_pi(theta)
    gs, pl = upd._surrogate(full, T, n)
    gs64, pl64 = prob.gradient(theta)
    np.testing.assert_allclose(gs, gs64, rtol=0, atol=2e-4 * np.abs(gs64).max())
    assert abs(pl - pl64) < 1e-5


@pytest.mark.parametrize("activation", ["leaky_relu", "tanh"])
@pytest.mark.parametrize("T,n", [(1, 100), (3, 1000), (2, 20000)])
def test_policy_mu_and_kl_gradient(cuda_device, activation, T, n):
    _check_mu_and_kl_gradient(cuda_device, DIMS, "fp32", activation, T, n, mu_atol=2e-5)


@pytest.mark.parametrize("kernel", ["fp32", "tensor_core"])
@pytest.mark.parametrize("obs_dim,act_dim", [(9, 7), (9, 5), (6, 3), (9, 6)])
@pytest.mark.parametrize("hidden", [(64, 64), (64, 64, 64), (80, 80, 80)], ids=["64x64", "64^3", "80^3"])
def test_policy_mu_and_kl_gradient_at_every_shape(cuda_device, hidden, obs_dim, act_dim, kernel):
    """The mean-only and the KL branches of every gradient kernel (ppo_grad_kernel at 64 x 64 9 -> 7, the generic fp32 one at
    the other shapes, the tensor-core one) at the reference's 80^3 and 64^3 networks and the run-time dims of RevoltLimited
    (9 -> 5), RevoltSimple (6 -> 3) and RevoltFinal without continuous angles (9 -> 6).  Batches: the reference's 4 x 400, a
    ragged 3 x 1037; 80^3 on tensor cores also 297 tiles, the two-group variant (296 tiles and fewer run the single-group one)."""
    dims = dict(obs_dim=obs_dim, act_dim=act_dim, hidden=hidden[0], n_hidden=len(hidden))
    batches = [(4, 400), (3, 1037)]
    if hidden == (80, 80, 80) and kernel == "tensor_core" and (obs_dim, act_dim) == (9, 7):
        batches.append((1, 297 * 128 - 5))
    for T, n in batches:
        _check_mu_and_kl_gradient(cuda_device, dims, kernel, "leaky_relu", T, n)


def test_hessian_vector_product_and_policy_update(cuda_device, dims=DIMS):
    import ml4ca_b200 as M
    T, n = 4, 8192
    ac, data, prob, theta, mu64 = _setup(cuda_device, T, n, seed=2, dims=dims)
    buf = M.GAEBuffer(dims["obs_dim"], dims["act_dim"], T, n, device=cuda_device)
    buf.obs_buf.copy_(data[0])
    buf.record_info(ac)
    full = data + [buf.log_std_buf, buf.mu_buf]
    upd = M.TRPOUpdater(ac)
    rng = np.random.default_rng(4)
    g64, _ = prob.gradient(theta)
    for v in (rng.normal(size=theta.size), g64):
        h = upd.hvp(full, T, n, theta, v)
        h64 = prob.hvp(theta, v, damping=0.1)
        assert np.linalg.norm(h - h64) < 3e-3 * np.linalg.norm(h64)
    assert torch.equal(upd._pi_params().cpu(), torch.as_tensor(theta.astype(np.float32)))   # hvp restores the parameters
    ref = TO.update(prob, theta)
    info = upd.update_policy(full, T, n)
    assert info["BacktrackIters"] == ref["backtrack_iters"]
    x, x64 = upd.last["x"], ref["x"]
    assert np.dot(x, x64) / (np.linalg.norm(x) * np.linalg.norm(x64)) > 0.999
    assert abs(upd.last["alpha"] / ref["alpha"] - 1) < 2e-2
    theta_new = upd._pi_params().double().cpu().numpy()
    step = np.linalg.norm(ref["theta"] - theta)
    # the parameters against the float64 update built the product's way (central differences of the KL gradient, radius 2e-3):
    # with three hidden layers the difference construction itself lands up to a few % of the step away from the exact update
    # (64^3 on this buffer: 2.4 % in float64, cosine 0.9997), so the exact one bounds them at two layers only
    ref_fd = TO.update(prob, theta, fd_radius=2e-3)
    assert ref_fd["backtrack_iters"] == ref["backtrack_iters"]
    assert step > 0 and np.linalg.norm(theta_new - ref_fd["theta"]) < 2e-2 * step
    if dims["n_hidden"] == 2:
        assert np.linalg.norm(theta_new - ref["theta"]) < 2e-2 * step
    assert info["KL"] <= 0.01 and info["DeltaLossPi"] < 0
    assert abs(info["KL"] - ref["kl"]) < 5e-2 * ref["kl"] and abs(info["LossPi"] - ref["pi_l_old"]) < 1e-5
    assert abs(info["DeltaLossPi"] - (ref["pi_l_new"] - ref["pi_l_old"])) < 5e-2 * abs(ref["pi_l_new"] - ref["pi_l_old"])
    # natural policy gradient: the full step, no line search
    upd._set_pi(theta)
    npg = M.TRPOUpdater(ac, algo='npg')
    info = npg.update_policy(full, T, n)
    np.testing.assert_allclose(npg._pi_params().double().cpu().numpy(),
                               (theta - npg.last["alpha"] * npg.last["x"]).astype(np.float32), rtol=0, atol=1e-7)
    assert "BacktrackIters" not in info


@pytest.mark.parametrize("hidden", [(64, 64, 64), (80, 80, 80)], ids=["64^3", "80^3"])
def test_hessian_vector_product_and_policy_update_at_three_hidden_layers(cuda_device, hidden):
    """The test above with the reference's shipped 64^3 and default 80^3 networks (generic fp32 kernel): same accepted line-search
    index, step cosine > 0.999, alpha within 2 %, parameters within 2 % of the step of the float64 central-difference update."""
    test_hessian_vector_product_and_policy_update(cuda_device, dict(obs_dim=9, act_dim=7, hidden=hidden[0], n_hidden=3))


@pytest.mark.parametrize("algo", ["trpo", "npg"])
def test_training_run_and_log_columns(cuda_device, tmp_path, algo):
    """trpo() end to end on a small batched env: every epoch respects the KL budget (trpo), the value loss falls, and
    progress.txt carries the reference's TRPO columns in its order (trpo.py:366-384)."""
    import ml4ca_b200 as M
    from ml4ca_b200.env import RevoltFinal, StandInHull
    env = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=2048, device=cuda_device, seed=3,
                      auto_reset=True)
    out = str(tmp_path / algo)
    ac, hist = M.trpo(env, steps_per_epoch=32, epochs=3, seed=1, algo=algo, train_v_iters=20,
                      logger_kwargs=dict(output_dir=out, exp_name=algo))
    for h in hist:
        assert np.isfinite([h["LossPi"], h["LossV"], h["KL"], h["DeltaLossPi"], h["DeltaLossV"]]).all()
        assert h["DeltaLossV"] < 0
        if algo == "trpo":
            assert h["KL"] <= 0.01 and h["DeltaLossPi"] <= 0 and 0 <= h["BacktrackIters"] <= 9
        else:
            assert h["KL"] < 0.05
    header = open(out + "/progress.txt").readline().rstrip("\n").split("\t")
    want = ["Epoch", "AverageEpRet", "StdEpRet", "MaxEpRet", "MinEpRet", "EpLen", "AverageVVals", "StdVVals", "MaxVVals",
            "MinVVals", "TotalEnvInteracts", "LossPi", "LossV", "DeltaLossPi", "DeltaLossV", "KL"]
    want += (["BacktrackIters"] if algo == "trpo" else []) + ["Time"]
    assert header == want
    import json
    cfg = json.load(open(out + "/config.json"))
    assert cfg["algo"] == algo and cfg["damping_coeff"] == 0.1 and cfg["cg_iters"] == 10


def test_tensor_core_kernel_option(cuda_device):
    """TRPOUpdater(kernel='tensor_core'): the KL-gradient passes of the CG solve on the tcgen05 kernel.  Stated accuracy: the
    Hessian-vector product within 2 % of the exact one (measured 0.2-0.3 %, tools/trpo_margins.py), step direction cosine
    > 0.998 (measured 0.9997-0.9999), step length within 2 %, the update inside the KL budget and improving the surrogate."""
    import ml4ca_b200 as M
    T, n = 4, 8192
    ac, data, prob, theta, mu64 = _setup(cuda_device, T, n, seed=2)
    buf = M.GAEBuffer(9, 7, T, n, device=cuda_device)
    buf.obs_buf.copy_(data[0])
    buf.record_info(ac)
    full = data + [buf.log_std_buf, buf.mu_buf]
    upd = M.TRPOUpdater(ac, kernel='tensor_core')
    upd._record_mu_tc(full, T, n)
    np.testing.assert_allclose(_flatten(upd._mu_tc.cpu().numpy()), mu64, rtol=0, atol=4e-3 * (1 + np.abs(mu64).max()))
    g0, kl0 = upd._kl(full, T, n, tensor_core=True)
    assert abs(kl0) < 1e-6                                       # d_kl(theta_old) = 0 with the kernel's own means
    g64, _ = prob.gradient(theta)
    h = upd.hvp(full, T, n, theta, g64, tensor_core=True)
    h64 = prob.hvp(theta, g64, damping=0.1)
    assert np.linalg.norm(h - h64) < 2e-2 * np.linalg.norm(h64)
    ref = TO.update(prob, theta)
    info = upd.update_policy(full, T, n)
    x, x64 = upd.last["x"], ref["x"]
    assert np.dot(x, x64) / (np.linalg.norm(x) * np.linalg.norm(x64)) > 0.998
    assert abs(upd.last["alpha"] / ref["alpha"] - 1) < 0.02
    assert info["KL"] <= 0.01 and info["DeltaLossPi"] < 0


def test_tensor_core_kernel_option_for_the_shipped_architecture(cuda_device):
    """kernel='tensor_core' with the reference's default 80 x 80 x 80 network: the KL-gradient passes run on the tcgen05 kernel
    templated on width and depth (csrc/ppo_update_tc.cu), checked against the float64 TRPO restatement on the same buffer: means
    within the fp16 tolerance, Hessian-vector product within 2 % of the exact one, and a whole TRPO update inside the KL budget
    that improves the surrogate.  65 536 samples: the two-group variant of the kernel."""
    import ml4ca_b200 as M
    T, n = 4, 16384
    rng = np.random.default_rng(3)
    dims = dict(obs_dim=9, act_dim=7, hidden=80, n_hidden=3)
    flat = MO.glorot_params(dims, seed=5)
    flat = (flat + rng.normal(size=flat.size).astype(np.float32) * 0.05).astype(np.float32)
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=flat, device=cuda_device)
    obs = torch.as_tensor((rng.normal(size=(T, 9, n)) * OBS_SCALE[None, :, None]).astype(np.float32), device=cuda_device)
    buf = M.GAEBuffer(9, 7, T, n, device=cuda_device)
    buf.obs_buf.copy_(obs)
    a, _, lp = ac.step(obs.permute(1, 0, 2).reshape(9, -1).contiguous(), deterministic=False, step=0)
    act = a.reshape(7, T, n).permute(1, 0, 2).contiguous()
    buf.record_info(ac)                                          # means of the old policy from the fp32 generic kernel
    mu_fp32 = buf.mu_buf.clone()
    eps = (act - mu_fp32) / torch.exp(buf.log_std_buf.reshape(1, 7, 1))
    adv = eps[:, 0, :] + 0.5 * torch.randn(T, n, device=cuda_device, generator=torch.Generator(device=cuda_device).manual_seed(1))
    adv = (adv - adv.mean()) / adv.std()
    data = [obs, act, adv.contiguous(), torch.zeros(T, n, device=cuda_device), lp.reshape(T, n).contiguous()]
    full = data + [buf.log_std_buf, buf.mu_buf]
    theta = flat[:TO.n_pi(dims)].astype(np.float64)
    ls = theta[-7:]
    f = lambda x: _flatten(x.cpu().numpy())
    prob = TO.Problem(dims, "leaky_relu", f(obs), f(act), adv.reshape(-1).cpu().numpy(), lp.reshape(-1).cpu().numpy(),
                      np.zeros((T * n, 7)), ls)
    mu64 = prob.mu(theta)
    prob.mu_old = torch.as_tensor(mu64)                          # d_kl = 0 at theta_old in float64 too
    upd = M.TRPOUpdater(ac, kernel='tensor_core')
    upd._record_mu_tc(full, T, n)
    np.testing.assert_allclose(f(upd._mu_tc), mu64, rtol=0, atol=6e-3 * (1 + np.abs(mu64).max()))   # three fp16 layers
    g0, kl0 = upd._kl(full, T, n, tensor_core=True)
    assert abs(kl0) < 1e-6
    assert torch.equal(upd._pi_params().cpu(), torch.as_tensor(theta.astype(np.float32)))
    v, _ = upd._surrogate(full, T, n)                            # the direction the CG solve starts from (as in the 64 x 64 test)
    h_tc = upd.hvp(full, T, n, theta, v, tensor_core=True)
    h64 = prob.hvp(theta, v, damping=0.1)
    assert np.linalg.norm(h_tc - h64) < 2e-2 * np.linalg.norm(h64)
    info = upd.update_policy(full, T, n)
    assert info["KL"] <= 0.01 and info["DeltaLossPi"] < 0


def test_training_run_of_the_shipped_architecture(cuda_device):
    """trpo() end to end with the reference's default 80 x 80 x 80 network at its batch size (4 envs x 400 steps): every epoch
    finite, inside the KL budget, and the line search never accepts a step that worsens the surrogate."""
    import ml4ca_b200 as M
    from ml4ca_b200.env import RevoltFinal, StandInHull
    env = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=4, device=cuda_device, seed=3, auto_reset=True)
    ac, hist = M.trpo(env, steps_per_epoch=400, epochs=2, seed=3, hidden_sizes=(80, 80, 80))
    assert ac.hidden_sizes == (80, 80, 80) and len(hist) == 2
    for h in hist:
        assert np.isfinite([h["LossPi"], h["LossV"], h["KL"], h["DeltaLossPi"], h["DeltaLossV"]]).all()
        assert h["KL"] <= 0.01 and h["DeltaLossPi"] <= 0
