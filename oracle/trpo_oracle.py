"""Float64 restatement of the reference's TRPO / NPG update (spinup/algos/tf1/trpo of src/rl/windows_workspace).

TEST INFRASTRUCTURE (see oracle/__init__.py).  TensorFlow 1 is not installable here, so the graph pieces are
restated with torch float64 autograd, each function citing the lines it follows:

  trpo/core.py:49-51   gaussian_likelihood
  trpo/core.py:52-60   diagonal_gaussian_kl(mu0, log_std0, mu1, log_std1)
  trpo/core.py:68-72   hessian_vector_product (gradient of <grad f, x>: double back-propagation, exact)
  trpo/core.py:88-100  mlp_gaussian_policy: d_kl = diagonal_gaussian_kl(mu, log_std, old_mu, old_log_std)
  trpo/trpo.py:236-247 ratio, pi_loss, flat gradient, damped hvp
  trpo/trpo.py:264-281 cg
  trpo/trpo.py:283-321 update(): x = cg(Hx, g), alpha, backtracking line search

Parameters are the flat vector of ml4ca_b200 (reference variable order); only the pi block [0, n_pi) moves.
Parity unpinned against TensorFlow itself (no TF1 here); the formulas are pinned to the source lines above and the
autograd engine supplies the derivatives.
"""
import numpy as np
import torch

EPS = 1e-8


def _pi_sizes(dims):
    """Layer widths of the pi net: [obs] + [H] * n_hidden + [act] (the pi block of mlp_oracle.unflatten)."""
    return [dims["obs_dim"]] + [dims["hidden"]] * dims["n_hidden"] + [dims["act_dim"]]


def n_pi(dims):
    """Size of the pi block: every (W [in, out], b [out]) of the pi net, then log_std [act]."""
    s = _pi_sizes(dims)
    return sum(s[i] * s[i + 1] + s[i + 1] for i in range(len(s) - 1)) + dims["act_dim"]


def _pi_net(theta, dims, obs, activation):
    """theta: torch float64 [n_pi]; obs [N, obs_dim] -> mu [N, act], log_std [act]."""
    sizes = _pi_sizes(dims)
    pos = [0]

    def take(*shape):
        k = int(np.prod(shape))
        t = theta[pos[0]:pos[0] + k].reshape(*shape)
        pos[0] += k
        return t

    layers = [(take(sizes[i], sizes[i + 1]), take(sizes[i + 1])) for i in range(len(sizes) - 1)]
    ls = take(dims["act_dim"])
    f = (lambda z: torch.where(z > 0, z, 0.2 * z)) if activation in ("leaky_relu", 1) else torch.tanh
    h = obs
    for W, b in layers[:-1]:
        h = f(h @ W + b)
    W, b = layers[-1]
    return h @ W + b, ls


def gaussian_likelihood(x, mu, log_std):
    pre = -0.5 * (((x - mu) / (torch.exp(log_std) + EPS)) ** 2 + 2 * log_std + np.log(2 * np.pi))
    return pre.sum(dim=1)


def diagonal_gaussian_kl(mu0, log_std0, mu1, log_std1):
    var0, var1 = torch.exp(2 * log_std0), torch.exp(2 * log_std1)
    pre = 0.5 * (((mu1 - mu0) ** 2 + var0) / (var1 + EPS) - 1) + log_std1 - log_std0
    return pre.sum(dim=1).mean()


class Problem(object):
    """One update's data: obs [N, obs], act [N, act], adv [N], logp_old [N], mu_old [N, act], log_std_old [act]."""

    def __init__(self, dims, activation, obs, act, adv, logp_old, mu_old, log_std_old):
        t = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float64))
        self.dims, self.activation = dims, activation
        self.obs, self.act, self.adv, self.logp_old = t(obs), t(act), t(adv), t(logp_old)
        self.mu_old, self.ls_old = t(mu_old), t(log_std_old)

    def mu(self, theta):
        with torch.no_grad():
            return _pi_net(torch.as_tensor(theta, dtype=torch.float64), self.dims, self.obs, self.activation)[0].numpy()

    def pi_loss(self, theta):                                          # trpo.py:236-237
        mu, ls = _pi_net(theta, self.dims, self.obs, self.activation)
        ratio = torch.exp(gaussian_likelihood(self.act, mu, ls) - self.logp_old)
        return -(ratio * self.adv).mean()

    def d_kl(self, theta):                                             # trpo/core.py:98
        mu, ls = _pi_net(theta, self.dims, self.obs, self.activation)
        return diagonal_gaussian_kl(mu, ls, self.mu_old, self.ls_old.expand_as(self.mu_old))

    def gradient(self, theta):                                         # trpo.py:244
        th = torch.tensor(np.asarray(theta, dtype=np.float64), requires_grad=True)
        loss = self.pi_loss(th)
        (g,) = torch.autograd.grad(loss, th)
        return g.numpy(), float(loss.detach())

    def kl_gradient(self, theta):
        th = torch.tensor(np.asarray(theta, dtype=np.float64), requires_grad=True)
        kl = self.d_kl(th)
        (g,) = torch.autograd.grad(kl, th)
        return g.numpy(), float(kl.detach())

    def hvp(self, theta, x, damping=0.0):                              # trpo/core.py:68-72, trpo.py:245-247
        th = torch.tensor(np.asarray(theta, dtype=np.float64), requires_grad=True)
        kl = self.d_kl(th)
        (g,) = torch.autograd.grad(kl, th, create_graph=True)
        xv = torch.as_tensor(np.asarray(x, dtype=np.float64))
        (h,) = torch.autograd.grad((g * xv).sum(), th)
        return h.numpy() + damping * np.asarray(x, dtype=np.float64)

    def evaluate(self, theta):
        with torch.no_grad():
            th = torch.as_tensor(np.asarray(theta, dtype=np.float64))
            return float(self.d_kl(th)), float(self.pi_loss(th))


def cg(Ax, b, cg_iters=10):
    """trpo.py:264-281: conjugate gradients from x = 0, a fixed number of steps, +1e-8 in the step-length denominator."""
    x = np.zeros_like(b)
    res, direction = b.copy(), b.copy()
    rr = np.dot(res, res)
    for _ in range(cg_iters):
        Ad = Ax(direction)
        step = rr / (np.dot(direction, Ad) + EPS)
        x += step * direction
        res -= step * Ad
        rr_next = np.dot(res, res)
        direction = res + (rr_next / rr) * direction
        rr = rr_next
    return x


def fd_hvp(prob, theta, x, radius, damping=0.0):
    """The Hessian-vector product as ml4ca_b200.trpo.TRPOUpdater.hvp builds it: a central difference of the KL gradient over
    +-radius along x (exact for quadratics; leaky-ReLU units that change branch inside the bracket perturb it)."""
    x = np.asarray(x, dtype=np.float64)
    e = radius / np.linalg.norm(x)
    return (prob.kl_gradient(theta + e * x)[0] - prob.kl_gradient(theta - e * x)[0]) / (2 * e) + damping * x


def update(prob, theta_old, target_kl=0.01, damping_coeff=0.1, cg_iters=10, backtrack_iters=10, backtrack_coeff=0.8,
           algo="trpo", fd_radius=None):
    """trpo.py:283-321 (policy part).  -> dict(theta, x, alpha, g, pi_l_old, pi_l_new, kl, backtrack_iters).
    fd_radius: the Hessian-vector products by fd_hvp instead of the exact double back-propagation of the reference."""
    theta_old = np.asarray(theta_old, dtype=np.float64)
    if fd_radius is None:
        Hx = lambda v: prob.hvp(theta_old, v, damping_coeff)
    else:
        Hx = lambda v: fd_hvp(prob, theta_old, v, fd_radius, damping_coeff)
    g, pi_l_old = prob.gradient(theta_old)
    x = cg(Hx, g, cg_iters)
    alpha = np.sqrt(2 * target_kl / (np.dot(x, Hx(x)) + EPS))
    out = dict(g=g, x=x, alpha=alpha, pi_l_old=pi_l_old)
    if algo == "npg":
        theta = theta_old - alpha * x
        kl, pi_l_new = prob.evaluate(theta)
        out.update(theta=theta, kl=kl, pi_l_new=pi_l_new, backtrack_iters=0)
        return out
    for j in range(backtrack_iters):
        theta = theta_old - alpha * x * backtrack_coeff ** j
        kl, pi_l_new = prob.evaluate(theta)
        if kl <= target_kl and pi_l_new <= pi_l_old:
            break
        if j == backtrack_iters - 1:
            theta = theta_old.copy()
            kl, pi_l_new = prob.evaluate(theta)
    out.update(theta=theta, kl=kl, pi_l_new=pi_l_new, backtrack_iters=j)
    return out
