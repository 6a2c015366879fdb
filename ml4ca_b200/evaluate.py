"""Evaluation harness: the shipped (or a freshly trained) policy inside the batched env, and the thesis' metrics.

Mirrors /root/reference/src/rl/windows_workspace/spinup/utils/test_policy.py (run_RL_policy :97-186: deterministic
action = mu, the fixed test poses of simtools.py:91-107, per-step records of observation, reward, NED pose and the
action vector) and the metric definitions of results/all_plots (IAE common.py:60-74, W* and IADC
box_test/plot_act.py:128-135,184-207,320-391).  Every env of the batch is one evaluation run; run k starts from fixed
test pose k mod 6.
"""
import numpy as np
import torch

from . import _lib

FIXED_THETAS = [0.0, np.pi / 4, np.pi / 2, np.pi, 5 * np.pi / 4, 3 * np.pi / 2]     # simtools.py:95
FIXED_ANGLES_DEG = [0.0, 0.0, -15.0, 15.0, 0.0, -15.0]                               # :96


def fixed_test_poses(n):
    """simtools.py:91-107 for runs 0..n-1 (pose k mod 6): -> eta [3, n] (N, E, yaw rad) on the r = 5 m circle."""
    k = np.arange(n) % len(FIXED_THETAS)
    ang = np.pi / 2 - np.asarray(FIXED_THETAS)[k]
    return np.stack([5 * np.sin(ang), 5 * np.cos(ang), np.deg2rad(np.asarray(FIXED_ANGLES_DEG)[k])])


def sensed(st):
    """The pose and velocity a controller receives from ``env.get_state()``: the measured values while the env has wave
    motion on (LF state plus waves, what a vessel's sensors report), else the state itself."""
    if "eta_measured" in st:
        return st["eta_measured"], st["nu_measured"]
    return st["eta"], st["nu"]


def in_loop_observer(env, observer):
    """The observer a controller acts on: the one attached to ``env`` (``Revolt.set_observer``), which the env steps and
    resets itself, else ``observer``.  -> (observer, attached).  A second observer next to an attached one is an error."""
    attached = getattr(env, "_observer", None)
    if attached is None:
        return observer, False
    if observer is not None and observer is not attached:
        raise ValueError("the env has an observer attached (set_observer); the controllers act on it, so a second "
                         "observer= cannot be passed")
    return attached, True


def run_RL_policy(env, ac, max_ep_len=None, new_ref=None, ref_change_at=None, integrator=False, observer=None):
    """test_policy.py:97-186 for every env of ``env`` at once (one episode each, no early stop: finished runs keep
    being recorded, ``done_at`` tells where the reference loop would have cut).  Returns a dict of device tensors:
    obs [T+1, obs, n], rew [T, n], eta [T+1, 3, n], thrust [T+1, 3, n], angles [T+1, 2, n], ref [T+1, 3, n], done_at [n],
    ep_ret [n], metrics [3, n] = IAE, W*, IADC.

    new_ref / ref_change_at: at step ``ref_change_at`` the env is stepped with a zero action and ``new_ref`` (test_policy.py
    :141-146).  The env takes the new set-point after that step (customEnv.py:131), so the observation the step returns is
    still relative to the old one: ``ref[s]`` is the set-point observation s was formed with, and a change at step k first
    shows in sample k + 2.  The policy's state assembly (integrator / observer) uses the set-point of its sample, and the
    IAE integrates |eta - ref| sample by sample.

    integrator=True: the thesis' ``RLintegral`` configuration.  The policy's three error rows come from the deployment
    node's state assembly with its body-frame integrator (ml4ca_ros_state, rl_allocator.py:252-273, one env step = h):
    the error plus an integral that starts 5 s after the vessel entered the 5 m / 140 deg zone.  ``obs`` keeps the env's
    own observation; the final integrator state is returned as ``integrator`` [3, n].  With wave motion on, the state
    assembly reads the measured pose and velocity (``sensed``); ``eta`` and the metrics keep the LF pose.

    observer: a ``DPObserver`` between the sensors and the policy.  It is reset on the measured pose after the env reset
    and stepped after every env step with the measured pose and the thrust and azimuths the step applied; the policy's
    rows 0-2 are then the deployment node's state assembly (ml4ca_ros_state, with or without the integrator) on the
    estimated pose eta^, rows 3-5 the estimated velocity nu^, rows 6-8 stay the env's.  ``eta_hat`` and ``bias_hat``
    [T+1, 3, n] are recorded; ``eta`` and the metrics keep the LF pose and the applied thrust.  On an env with an attached
    observer (``Revolt.set_observer``) that observer is used: the env resets and steps it, and the policy input without
    the integrator is the env's observation, which is already formed from the estimates.  Passing another observer then
    raises ValueError."""
    observer, attached = in_loop_observer(env, observer)
    n, dev = env.num_envs, env.device
    T = int(max_ep_len if max_ep_len is not None else env.max_ep_len)
    eta0 = fixed_test_poses(n)
    o = env.reset(**{'Hull.PosNED': eta0[0:2], 'Hull.PosAttitude': np.stack([np.zeros(n), np.zeros(n), eta0[2]]),
                     'Hull.VelocityNu': np.zeros((6, n))})
    o = torch.as_tensor(o, dtype=torch.float32, device=dev).reshape(env.num_states, n)
    f = dict(dtype=torch.float32, device=dev)
    rec = {"obs": torch.empty(T + 1, env.num_states, n, **f), "rew": torch.zeros(T, n, **f),
           "eta": torch.empty(T + 1, 3, n, **f), "thrust": torch.zeros(T + 1, 3, n, **f),
           "angles": torch.zeros(T + 1, 2, n, **f), "ref": torch.empty(T + 1, 3, n, **f)}
    done_at = torch.full((n,), T, dtype=torch.int32, device=dev)
    st = env.get_state()
    rec["obs"][0], rec["eta"][0], rec["angles"][0], rec["ref"][0] = o, st["eta"], st["angles"][1:3], env._ref
    integ = t_inside = None
    if integrator:
        integ, t_inside = torch.zeros(3, n, **f), torch.zeros(n, **f)
    if integrator or observer is not None:
        prev_u, ros = torch.zeros(6, n, **f), torch.empty(9, n, **f)       # ROS-order previous thrust: rows 6-8 unused here
    if observer is not None:
        rec["eta_hat"], rec["bias_hat"] = torch.empty(T + 1, 3, n, **f), torch.empty(T + 1, 3, n, **f)
        if not attached:
            observer.reset(sensed(st)[0])
        rec["eta_hat"][0], rec["bias_hat"][0] = observer.eta_hat, observer.bias_hat

    def policy_input(o, st, ref):
        if not integrator and (observer is None or attached):
            return o
        eta_s, nu_s = sensed(st) if observer is None else (observer.eta_hat.contiguous(), observer.nu_hat.contiguous())
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().ml4ca_ros_state(n, _lib.ptr(eta_s), _lib.ptr(nu_s), _lib.ptr(ref), _lib.ptr(prev_u),
                                                  _lib.ptr(integ), _lib.ptr(t_inside), float(env.dt), _lib.ptr(ros),
                                                  _lib.current_stream()), "ml4ca_ros_state")
        x = o.clone()
        x[0:3] = ros[0:3]
        if observer is not None:
            x[3:6] = nu_s
        return x
    for t in range(T):
        a = ac.get_action(policy_input(o, st, rec["ref"][t]))                # deterministic action = mu (:90-93)
        rec["ref"][t + 1] = env._ref                                         # the set-point the step's observation is formed with
        if ref_change_at is not None and t == ref_change_at and new_ref is not None:
            o, r, d, _ = env.step(torch.zeros_like(a), new_ref=new_ref)      # :141-146
        else:
            o, r, d, _ = env.step(a)
        st = env.get_state()
        rec["obs"][t + 1], rec["rew"][t], rec["eta"][t + 1] = o, r, st["eta"]
        rec["thrust"][t + 1], rec["angles"][t + 1] = st["prev_thrust"], st["angles"][1:3]
        if observer is not None:
            if not attached:
                observer.step(sensed(st)[0], st["prev_thrust"], st["angles"])
            rec["eta_hat"][t + 1], rec["bias_hat"][t + 1] = observer.eta_hat, observer.bias_hat
        first = d & (done_at == T)
        done_at = torch.where(first, torch.full_like(done_at, t + 1), done_at)
    rec["done_at"] = done_at
    steps = torch.arange(T, device=dev)[:, None]
    rec["ep_ret"] = (rec["rew"] * (steps < done_at[None, :])).sum(dim=0)
    # IAE depends on eta - ref only: the per-sample error against a zero set-point is the metric of a varying set-point
    rec["metrics"] = metrics(rec["eta"] - rec["ref"], torch.zeros(3, n, **f), rec["thrust"], rec["angles"], env.dt)
    if integrator:
        rec["integrator"] = integ
    return rec


def run_allocator(env, method="qp", max_ep_len=None, observer=None):
    """The classical DP pipeline in the same batched env: PID on the body-frame error (ml4ca_pinv_pid) -> thrust
    allocation by the SLSQP-equivalent kernel (``method='qp'``, QPTA.tau_controller_callback_func) or the fixed-matrix
    pseudoinverse (``'pinv'``) -> env step.  Same records and metrics as run_RL_policy: with it, the thesis' comparison
    RL vs QP vs IPI (results/all_plots) runs for thousands of poses at once.  With wave motion on, the PID acts on the
    measured pose and velocity (``sensed``); ``eta`` and the metrics keep the LF pose.

    observer: a ``DPObserver`` between the sensors and the PID, as in run_RL_policy: the PID acts on (eta^, nu^); the
    records gain ``eta_hat`` and ``bias_hat`` [T+1, 3, n].  On an env with an attached observer that observer is used, as
    in run_RL_policy."""
    observer, attached = in_loop_observer(env, observer)
    from .pinv import pinv_pid
    from .qp_allocator import QPTA
    n, dev = env.num_envs, env.device
    assert env.name == 'revoltfinal', "the allocators command two rotating stern azimuths + the fixed bow thruster"
    T = int(max_ep_len if max_ep_len is not None else env.max_ep_len)
    eta0 = fixed_test_poses(n)
    o = env.reset(**{'Hull.PosNED': eta0[0:2], 'Hull.PosAttitude': np.stack([np.zeros(n), np.zeros(n), eta0[2]]),
                     'Hull.VelocityNu': np.zeros((6, n))})
    f = dict(dtype=torch.float32, device=dev)
    rec = {"rew": torch.zeros(T, n, **f), "eta": torch.empty(T + 1, 3, n, **f), "thrust": torch.zeros(T + 1, 3, n, **f),
           "angles": torch.zeros(T + 1, 2, n, **f)}
    st = env.get_state()
    rec["eta"][0], rec["angles"][0] = st["eta"], st["angles"][1:3]
    if observer is not None:
        rec["eta_hat"], rec["bias_hat"] = torch.empty(T + 1, 3, n, **f), torch.empty(T + 1, 3, n, **f)
        if not attached:
            observer.reset(sensed(st)[0])
        rec["eta_hat"][0], rec["bias_hat"][0] = observer.eta_hat, observer.bias_hat
    integ = torch.zeros(3, n, **f)
    qp = QPTA(num_envs=n, device=dev) if method == "qp" else None
    action = torch.empty(env.num_actions, n, **f)
    ref = env._ref.clone()
    # The SLSQP programme only admits demands its rate limits can follow (|df| <= 5, 5, 2 N per call): on the vessel the
    # reference filter feeds it smooth demands.  Stand-in: the demand is the wrench the thrusters deliver now plus the
    # PID's request clipped to +-[4, 2, 2] -- the neighbourhood law of BASELINE config 1 (99.7 % success with the
    # reference solver).
    slew = torch.tensor([[4.0], [2.0], [2.0]], **f)
    lx, ly = (-1.12, -1.12, 1.08), (-0.15, 0.15, 0.0)            # qp_allocator.py:69-70

    def delivered(prev):                                           # B(alpha) f of the allocator's current state
        f0, f1, f2, a0, a1 = prev
        c0, s0, c1, s1 = torch.cos(a0), torch.sin(a0), torch.cos(a1), torch.sin(a1)
        return torch.stack([f0 * c0 + f1 * c1, f0 * s0 + f1 * s1 + f2,
                            f0 * (lx[0] * s0 - ly[0] * c0) + f1 * (lx[1] * s1 - ly[1] * c1) + f2 * lx[2]])
    trust = torch.ones(n, **f)     # per-run scale of the clip: halved when the programme is infeasible (the allocator then
    for t in range(T):             # holds its state, qp_allocator.py:267-269), restored step by step when it succeeds
        eta_s, nu_s = sensed(st) if observer is None else (observer.eta_hat.contiguous(), observer.nu_hat.contiguous())
        n_pct, alpha, tau = pinv_pid(eta_s, nu_s, ref, integ, return_tau=True)
        if qp is not None:
            now = delivered(qp._prev)
            lim = slew * trust[None, :]
            qp.tau_controller_callback_func(now + torch.minimum(torch.maximum(tau - now, -lim), lim))
            ok = (qp.last_status & 1).bool()
            trust = torch.where(ok, (trust * 2).clamp(max=1.0), trust * 0.5)
            n_pct, alpha = qp.last_output[0:3].contiguous(), qp.last_output[3:5].contiguous()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().ml4ca_alloc_to_action(n, int(env.cont_ang), float(env.real_action_bounds[3]), _lib.ptr(n_pct),
                                                        _lib.ptr(alpha), _lib.ptr(action), _lib.current_stream()),
                       "ml4ca_alloc_to_action")
        o, r, d, _ = env.step(action)
        st = env.get_state()
        rec["rew"][t], rec["eta"][t + 1] = r, st["eta"]
        rec["thrust"][t + 1], rec["angles"][t + 1] = st["prev_thrust"], st["angles"][1:3]
        if observer is not None:
            if not attached:
                observer.step(sensed(st)[0], st["prev_thrust"], st["angles"])
            rec["eta_hat"][t + 1], rec["bias_hat"][t + 1] = observer.eta_hat, observer.bias_hat
    rec["ep_ret"] = rec["rew"].sum(dim=0)
    rec["metrics"] = metrics(rec["eta"], ref, rec["thrust"], rec["angles"], env.dt)
    return rec


def metrics(eta, ref, thrust, angles, dt):
    """IAE, W*, IADC per run (ml4ca_eval_metrics): eta [T, 3, n], ref [3, n], thrust [T, 3, n], angles [T, 2, n]."""
    T, _, n = eta.shape
    out = torch.empty(3, n, dtype=torch.float32, device=eta.device)
    eta, ref, thrust, angles = eta.contiguous(), ref.contiguous(), thrust.contiguous(), angles.contiguous()
    with torch.cuda.device(eta.device):
        _lib.check(_lib.lib().ml4ca_eval_metrics(n, T, float(dt), _lib.ptr(eta), _lib.ptr(ref), _lib.ptr(thrust),
                                                 _lib.ptr(angles), _lib.ptr(out), _lib.current_stream()), "ml4ca_eval_metrics")
    return out
