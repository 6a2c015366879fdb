"""The float64 TRPO restatement (oracle/trpo_oracle.py) checked for internal consistency on the CPU: the exact
Hessian-vector product of d_kl (double back-propagation, trpo/core.py:68-72) against a central difference of the
KL gradient -- the construction the CUDA path uses -- and the closed form of the log_std block; its pi net against the
actor forward of oracle/mlp_oracle.py.  Every network shape the kernels serve: 64 x 64, 64^3 and 80^3 (the reference's
default and its shipped models), and the run-time observation / action dims of the other env classes."""
import numpy as np
import pytest
import torch

from oracle import mlp_oracle as MO
from oracle import trpo_oracle as TO

SHAPES = [dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=2), dict(obs_dim=9, act_dim=7, hidden=64, n_hidden=3),
          dict(obs_dim=9, act_dim=7, hidden=80, n_hidden=3), dict(obs_dim=9, act_dim=5, hidden=64, n_hidden=3)]
SHAPE_IDS = ["64x64", "64^3", "80^3", "64^3-9to5"]     # the consistency tests below run 64x64 themselves, the rest here
OBS_SCALE = np.array([2, 2, .3, .5, .1, .2, .5, .5, .5])


def make_problem(dims=SHAPES[0], N=400, seed=0, activation="leaky_relu"):
    O, A = dims["obs_dim"], dims["act_dim"]
    rng = np.random.default_rng(seed)
    flat = MO.glorot_params(dims, 3).astype(np.float64)
    flat = flat + rng.normal(size=flat.size) * 0.05
    theta = flat[:TO.n_pi(dims)].copy()
    obs = rng.normal(size=(N, O)) * OBS_SCALE[:O]
    ls = theta[-A:]
    prob0 = TO.Problem(dims, activation, obs, np.zeros((N, A)), np.zeros(N), np.zeros(N), np.zeros((N, A)), ls)
    mu = prob0.mu(theta)
    act = mu + rng.normal(size=mu.shape) * np.exp(ls)
    logp = MO.gaussian_likelihood(act, mu, ls)
    adv = rng.normal(size=N)
    adv = (adv - adv.mean()) / adv.std()
    return TO.Problem(dims, activation, obs, act, adv, logp, mu, ls), theta


@pytest.mark.parametrize("hidden", [(64, 64), (64, 64, 64), (80, 80, 80)])
@pytest.mark.parametrize("obs_dim,act_dim", [(9, 7), (9, 5), (6, 3), (9, 6)])
@pytest.mark.parametrize("activation", ["leaky_relu", "tanh"])
def test_pi_net_equals_the_actor_forward(hidden, obs_dim, act_dim, activation):
    """n_pi = the pi block plus log_std of mlp_oracle.unflatten, and _pi_net's means = mlp_oracle.forward's mu."""
    dims = dict(obs_dim=obs_dim, act_dim=act_dim, hidden=hidden[0], n_hidden=len(hidden))
    flat = MO.glorot_params(dims, 3).astype(np.float64)
    flat = flat + np.random.default_rng(1).normal(size=flat.size) * 0.05           # non-zero biases
    pi, log_std, _ = MO.unflatten(flat, dims)
    assert TO.n_pi(dims) == sum(W.size + b.size for W, b in pi) + log_std.size
    obs = np.random.default_rng(2).normal(size=(obs_dim, 300)) * OBS_SCALE[:obs_dim, None]
    mu, ls = TO._pi_net(torch.as_tensor(flat[:TO.n_pi(dims)]), dims, torch.as_tensor(obs.T), activation)
    np.testing.assert_allclose(mu.numpy().T, MO.forward(flat, dims, obs, activation)["mu"], rtol=0, atol=1e-12)
    np.testing.assert_array_equal(ls.numpy(), log_std)


def test_kl_is_zero_with_zero_gradient_at_theta_old(dims=SHAPES[0]):
    prob, theta = make_problem(dims)
    g, kl = prob.kl_gradient(theta)
    assert abs(kl) < 1e-6 and np.abs(g).max() < 1e-6          # the 1e-8 EPS of trpo/core.py:58 leaves ~1e-8 / var per action


def test_exact_hvp_equals_central_difference_of_kl_gradient(dims=SHAPES[0]):
    # three hidden layers carry more units that can change branch inside the bracket: the reference's 4 x 400 batch keeps
    # them inside the same bound (80^3 along the gradient, measured: 3.1e-3 at 400 samples, 1.5e-3 at 1600)
    prob, theta = make_problem(dims, N=400 if dims["n_hidden"] == 2 else 1600)
    rng = np.random.default_rng(1)
    for v in (rng.normal(size=theta.size), prob.gradient(theta)[0]):
        h = prob.hvp(theta, v)
        fd = TO.fd_hvp(prob, theta, v, 2e-3)             # fd_radius of ml4ca_b200.trpo.TRPOUpdater
        # piecewise-linear units that change branch inside the +-e v bracket bound the agreement (error ~ sqrt(radius / N))
        assert np.linalg.norm(fd - h) < 3e-3 * np.linalg.norm(h)
    # log_std block of the Hessian at theta_old: d2/dls2 [0.5 var / (var_old + EPS) - ls] = 2 on the diagonal
    e7 = np.zeros(theta.size); e7[-3] = 1.0
    h = prob.hvp(theta, e7)
    assert abs(h[-3] - 2.0) < 1e-6 and np.abs(np.delete(h, theta.size - 3)).max() < 1e-9


def test_update_respects_the_trust_region_and_improves_the_surrogate(dims=SHAPES[0]):
    prob, theta = make_problem(dims)
    out = TO.update(prob, theta)
    assert out["kl"] <= 0.01 and out["pi_l_new"] <= out["pi_l_old"]
    assert out["backtrack_iters"] < 9 and np.linalg.norm(out["theta"] - theta) > 0
    # the solve: x ~ (H + damping)^-1 g after 10 CG iterations -> residual well below |g|
    r = prob.hvp(theta, out["x"], 0.1) - out["g"]
    assert np.linalg.norm(r) < 0.5 * np.linalg.norm(out["g"])
    npg = TO.update(prob, theta, algo="npg")
    np.testing.assert_allclose(npg["theta"], theta - npg["alpha"] * npg["x"])


@pytest.mark.parametrize("dims", SHAPES[1:], ids=SHAPE_IDS[1:])
def test_consistency_at_the_other_network_shapes(dims):
    """The three consistency checks above at 64^3, 80^3 and 64^3 with the 9 -> 5 dims of RevoltLimited."""
    test_kl_is_zero_with_zero_gradient_at_theta_old(dims)
    test_exact_hvp_equals_central_difference_of_kl_gradient(dims)
    test_update_respects_the_trust_region_and_improves_the_surrogate(dims)


def test_product_cg_equals_oracle_cg_and_solves_spd_systems():
    """ml4ca_b200.trpo.TRPOUpdater.cg (host logic, no GPU needed) against the restatement of trpo.py:264-281 and against
    a direct solve: n iterations of conjugate gradients solve an n x n SPD system."""
    import types
    from ml4ca_b200.trpo import TRPOUpdater
    rng = np.random.default_rng(0)
    A = rng.normal(size=(12, 12))
    A = np.eye(12) + 0.3 * (A @ A.T) / 12.0          # well conditioned: 12 steps reach the solution in floating point
    b = rng.normal(size=12)
    for iters in (3, 12):
        me = types.SimpleNamespace(cg_iters=iters)
        x_prod = TRPOUpdater.cg(me, lambda v: A @ v, b.copy())
        x_orac = TO.cg(lambda v: A @ v, b.copy(), iters)
        np.testing.assert_allclose(x_prod, x_orac, rtol=1e-12, atol=1e-14)
    # the reference's +1e-8 in the step-length denominator damps the last steps: the solve stalls around 1e-5
    np.testing.assert_allclose(x_prod, np.linalg.solve(A, b), rtol=0, atol=1e-4)
