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


def box_test_schedule(side=5.0, yaw_deg=-45.0, hold_s=60.0, dt=0.2):
    """The four-corner DP box test as a set-point schedule -> (steps [7] int, setpoints [7, 3] (N m, E m, yaw rad)).

    On station at (0, 0, 0), then pure surge to (side, 0, 0), pure sway to (side, side, 0), pure yaw to
    (side, side, yaw), combined surge and sway to (0, side, yaw), and all three back to (0, 0, 0); the start and every leg
    are held ``hold_s``.  The last entry marks the end of the run (steps[-1] = 6 holds, the set-point of the final
    sample), so ``run_allocator`` / ``run_RL_policy`` run exactly the test by default.

    DECLARED, not pinned: the reference's own box-test schedule (results/all_plots/box_test/plot_pos.py) is not available
    to this build; this is the usual four-corner DP test."""
    k = int(round(hold_s / dt))
    y = float(np.deg2rad(yaw_deg))
    sp = np.array([[0.0, 0.0, 0.0], [side, 0.0, 0.0], [side, side, 0.0], [side, side, y], [0.0, side, y], [0.0, 0.0, 0.0],
                   [0.0, 0.0, 0.0]])
    return np.arange(len(sp), dtype=np.int64) * k, sp


class _Guidance(object):
    """The set-point side of an evaluation run with a schedule: s(t), the last entry with steps <= t, and the reference the
    controllers track, r(t) = s(t), or with a reference model r(t) = eta_d(t) (with v_d(t) for the PID's feed-forward).
    ``advance(t)`` moves the reference to r(t + 1) (the model steps once on s(t)) and hands it to the env (set_ref).

    With the model attached to the env (``attached``), the env steps and resets it: ``advance(t)`` only hands s(t) to the
    env, and ``stepped(t)`` reads r(t + 1) and v_d(t + 1) from the model after the env step.  Without a schedule an attached
    model guides the fixed-test-pose runs to the env's set-point: s(t) is that set-point throughout."""

    def __init__(self, env, schedule, reference_model, max_ep_len, attached=False):
        n, dev = env.num_envs, env.device
        self.fixed = schedule is None
        if self.fixed:
            schedule = (np.zeros(1, dtype=np.int64), env._ref.clone()[None])
            max_ep_len = max_ep_len if max_ep_len is not None else env.max_ep_len
        steps, sp = schedule
        steps = np.asarray(steps).reshape(-1)
        if steps.size == 0 or int(steps[0]) != 0 or np.any(np.diff(steps) <= 0):
            raise ValueError("schedule steps must start at 0 and be strictly increasing")
        sp = torch.as_tensor(sp, dtype=torch.float32, device=dev)
        if sp.dim() == 2 and sp.shape == (steps.size, 3):
            sp = sp[:, :, None].expand(steps.size, 3, n)
        elif sp.shape != (steps.size, 3, n):
            raise ValueError("schedule set-points must be [K, 3] or [K, 3, num_envs] for K = len(steps)")
        self.sp = sp.contiguous()
        if reference_model is not None and (reference_model.num_envs != n or
                                            abs(reference_model.step_dt - float(env.dt)) > 1e-6 * float(env.dt)):
            raise ValueError("the reference model's num_envs and step_dt must match the env's")
        self.T = int(max_ep_len if max_ep_len is not None else steps[-1])
        if self.T < 1:
            raise ValueError("the run needs at least one step: give max_ep_len or a schedule whose last step is > 0")
        self.idx = np.searchsorted(steps, np.arange(self.T + 1), side="right") - 1
        self.env, self.model, self.attached = env, reference_model, attached

    def s(self, t):
        return self.sp[int(self.idx[t])]

    def r(self):
        """The reference the env's observation is formed with now."""
        return self.model.eta_d.clone() if self.attached else self.env._ref.clone()

    def start(self, rec):
        """r(0) = s(0): the env's set-point before the reset, the model reset on it (an attached model is reset by the
        env's reset_to).  -> the start pose [3, n] numpy: s(0), or the fixed test poses without a schedule."""
        s0 = self.s(0)
        self.env.set_ref(s0)
        f = dict(dtype=torch.float32, device=self.env.device)
        T, n = self.T, self.env.num_envs
        rec["setpoint"] = torch.empty(T + 1, 3, n, **f)
        rec["setpoint"][0] = s0
        if self.model is not None:
            if not self.attached:
                self.model.reset(s0)
            rec["v_d"] = torch.empty(T + 1, 3, n, **f)
        return fixed_test_poses(n) if self.fixed else s0.double().cpu().numpy()

    def started(self, rec):
        """After the env reset: v_d(0)."""
        if self.model is not None:
            rec["v_d"][0] = self.model.v_d

    def advance(self, t, rec):
        if self.attached:
            self.env.set_ref(self.s(t))
        elif self.model is not None:
            self.model.step(self.s(t))
            self.env.set_ref(self.model.eta_d.clone())
            rec["v_d"][t + 1] = self.model.v_d
        else:
            self.env.set_ref(self.s(t + 1))
        rec["setpoint"][t + 1] = self.s(t + 1)

    def stepped(self, t, rec):
        """After the env step of step t: r(t + 1) and v_d(t + 1) of an attached model."""
        if self.attached:
            rec["ref"][t + 1] = self.model.eta_d
            rec["v_d"][t + 1] = self.model.v_d


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


def in_loop_reference_model(env, reference_model):
    """The reference model a run follows: the one attached to ``env`` (``Revolt.set_reference_model``), which the env steps
    and resets itself, else ``reference_model``.  -> (model, attached).  A second model next to an attached one is an
    error."""
    attached = getattr(env, "_refmodel", None)
    if attached is None:
        return reference_model, False
    if reference_model is not None and reference_model is not attached:
        raise ValueError("the env has a reference model attached (set_reference_model); the run follows it, so a second "
                         "reference_model= cannot be passed")
    return attached, True


def run_RL_policy(env, ac, max_ep_len=None, new_ref=None, ref_change_at=None, integrator=False, observer=None,
                  schedule=None, reference_model=None):
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
    raises ValueError.

    schedule = (steps [K], setpoints [K, 3] or [K, 3, n]): a set-point schedule such as ``box_test_schedule()``; s(t) is
    the entry of the last step <= t, steps ascend strictly from 0, T defaults to steps[-1].  Every run then starts at
    rest at s(0) instead of the fixed test poses.  The controller tracks r(t): s(t), or with ``reference_model`` (a
    ``ReferenceModel`` of the env's num_envs and step_dt, reset on s(0)) its eta_d(t).  In step t the policy acts on
    observation t, formed with r(t), then the reference advances to r(t + 1) (the model steps once on s(t)), the env
    takes it (set_ref) and steps: a schedule change at step k first shows in sample k.  The state assembly uses r(t).
    Records gain ``setpoint`` [T+1, 3, n] (s), ``ref`` is r, and with a model ``v_d`` [T+1, 3, n]; the IAE integrates
    against ``setpoint``, so runs with and without a reference model are scored against the same command.  A schedule
    together with new_ref / ref_change_at, bad steps, set-points of the wrong shape or a model that does not match the
    env raise ValueError; so does a reference model without a schedule.

    On an env with an attached reference model (``Revolt.set_reference_model``) that model is used: the env resets and
    steps it, and ``ref`` / ``v_d`` are read from it after each step; the records and metrics are those of the same run
    with ``reference_model=`` on a plain env.  Passing another model then raises ValueError.  Without a schedule the
    attached model guides the fixed-test-pose runs to the env's set-point: the records gain ``setpoint`` and the IAE is
    scored against it; new_ref / ref_change_at then raise ValueError."""
    observer, attached = in_loop_observer(env, observer)
    n, dev = env.num_envs, env.device
    plan = _plan(env, schedule, reference_model, max_ep_len)
    if plan is not None and (new_ref is not None or ref_change_at is not None):
        raise ValueError("a schedule (or an attached reference model) replaces new_ref / ref_change_at: pass one or the other")
    T = plan.T if plan is not None else int(max_ep_len if max_ep_len is not None else env.max_ep_len)
    rec = {}
    eta0 = plan.start(rec) if plan is not None else fixed_test_poses(n)
    o = env.reset(**{'Hull.PosNED': eta0[0:2], 'Hull.PosAttitude': np.stack([np.zeros(n), np.zeros(n), eta0[2]]),
                     'Hull.VelocityNu': np.zeros((6, n))})
    o = torch.as_tensor(o, dtype=torch.float32, device=dev).reshape(env.num_states, n)
    f = dict(dtype=torch.float32, device=dev)
    rec.update({"obs": torch.empty(T + 1, env.num_states, n, **f), "rew": torch.zeros(T, n, **f),
                "eta": torch.empty(T + 1, 3, n, **f), "thrust": torch.zeros(T + 1, 3, n, **f),
                "angles": torch.zeros(T + 1, 2, n, **f), "ref": torch.empty(T + 1, 3, n, **f)})
    done_at = torch.full((n,), T, dtype=torch.int32, device=dev)
    st = env.get_state()
    rec["obs"][0], rec["eta"][0], rec["angles"][0] = o, st["eta"], st["angles"][1:3]
    rec["ref"][0] = plan.r() if plan is not None else env._ref
    if plan is not None:
        plan.started(rec)
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
        if plan is not None:
            plan.advance(t, rec)
        rec["ref"][t + 1] = env._ref                                         # the set-point the step's observation is formed with
        if ref_change_at is not None and t == ref_change_at and new_ref is not None:
            o, r, d, _ = env.step(torch.zeros_like(a), new_ref=new_ref)      # :141-146
        else:
            o, r, d, _ = env.step(a)
        if plan is not None:
            plan.stepped(t, rec)
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
    cmd = rec["setpoint"] if plan is not None else rec["ref"]
    rec["metrics"] = metrics(rec["eta"] - cmd, torch.zeros(3, n, **f), rec["thrust"], rec["angles"], env.dt)
    if integrator:
        rec["integrator"] = integ
    return rec


def _plan(env, schedule, reference_model, max_ep_len):
    reference_model, attached = in_loop_reference_model(env, reference_model)
    if schedule is None and not attached:
        if reference_model is not None:
            raise ValueError("a reference model needs a schedule to filter")
        return None
    return _Guidance(env, schedule, reference_model, max_ep_len, attached)


def run_allocator(env, method="qp", max_ep_len=None, observer=None, schedule=None, reference_model=None):
    """The classical DP pipeline in the same batched env: PID on the body-frame error (ml4ca_pinv_pid) -> thrust
    allocation by the SLSQP-equivalent kernel (``method='qp'``, QPTA.tau_controller_callback_func) or the fixed-matrix
    pseudoinverse (``'pinv'``) -> env step.  Same records and metrics as run_RL_policy: with it, the thesis' comparison
    RL vs QP vs IPI (results/all_plots) runs for thousands of poses at once.  With wave motion on, the PID acts on the
    measured pose and velocity (``sensed``); ``eta`` and the metrics keep the LF pose.

    observer: a ``DPObserver`` between the sensors and the PID, as in run_RL_policy: the PID acts on (eta^, nu^); the
    records gain ``eta_hat`` and ``bias_hat`` [T+1, 3, n].  On an env with an attached observer that observer is used, as
    in run_RL_policy.

    schedule / reference_model: as in run_RL_policy.  The PID acts on r(t), and with a reference model it also gets
    v_d(t) as velocity feed-forward (``pinv_pid(nu_d=)``).  Records gain ``setpoint``, ``ref`` (r) [T+1, 3, n], with a
    model ``v_d``, and for ``method='qp'`` ``demand_clipped`` [T, n] (bool: the +-[4, 2, 2] demand clip below bound in
    some DOF at that step).  An attached reference model is used as in run_RL_policy; the PID's feed-forward then reads
    v_d from it."""
    observer, attached = in_loop_observer(env, observer)
    from .pinv import pinv_pid
    from .qp_allocator import QPTA
    n, dev = env.num_envs, env.device
    assert env.name == 'revoltfinal', "the allocators command two rotating stern azimuths + the fixed bow thruster"
    plan = _plan(env, schedule, reference_model, max_ep_len)
    T = plan.T if plan is not None else int(max_ep_len if max_ep_len is not None else env.max_ep_len)
    rec = {}
    eta0 = plan.start(rec) if plan is not None else fixed_test_poses(n)
    o = env.reset(**{'Hull.PosNED': eta0[0:2], 'Hull.PosAttitude': np.stack([np.zeros(n), np.zeros(n), eta0[2]]),
                     'Hull.VelocityNu': np.zeros((6, n))})
    f = dict(dtype=torch.float32, device=dev)
    rec.update({"rew": torch.zeros(T, n, **f), "eta": torch.empty(T + 1, 3, n, **f),
                "thrust": torch.zeros(T + 1, 3, n, **f), "angles": torch.zeros(T + 1, 2, n, **f)})
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
    if plan is not None:
        rec["ref"] = torch.empty(T + 1, 3, n, **f)
        rec["ref"][0] = plan.r()
        plan.started(rec)
        if qp is not None:
            rec["demand_clipped"] = torch.empty(T, n, dtype=torch.bool, device=dev)
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
        if plan is None:
            n_pct, alpha, tau = pinv_pid(eta_s, nu_s, ref, integ, return_tau=True)
        else:
            nu_d = rec["v_d"][t] if "v_d" in rec else None
            n_pct, alpha, tau = pinv_pid(eta_s, nu_s, rec["ref"][t], integ, return_tau=True, nu_d=nu_d)
        if qp is not None:
            now = delivered(qp._prev)
            lim = slew * trust[None, :]
            if plan is not None:
                rec["demand_clipped"][t] = ((tau - now).abs() > lim).any(dim=0)
            qp.tau_controller_callback_func(now + torch.minimum(torch.maximum(tau - now, -lim), lim))
            ok = (qp.last_status & 1).bool()
            trust = torch.where(ok, (trust * 2).clamp(max=1.0), trust * 0.5)
            n_pct, alpha = qp.last_output[0:3].contiguous(), qp.last_output[3:5].contiguous()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().ml4ca_alloc_to_action(n, int(env.cont_ang), float(env.real_action_bounds[3]), _lib.ptr(n_pct),
                                                        _lib.ptr(alpha), _lib.ptr(action), _lib.current_stream()),
                       "ml4ca_alloc_to_action")
        if plan is not None:
            plan.advance(t, rec)
            rec["ref"][t + 1] = env._ref
        o, r, d, _ = env.step(action)
        if plan is not None:
            plan.stepped(t, rec)
        st = env.get_state()
        rec["rew"][t], rec["eta"][t + 1] = r, st["eta"]
        rec["thrust"][t + 1], rec["angles"][t + 1] = st["prev_thrust"], st["angles"][1:3]
        if observer is not None:
            if not attached:
                observer.step(sensed(st)[0], st["prev_thrust"], st["angles"])
            rec["eta_hat"][t + 1], rec["bias_hat"][t + 1] = observer.eta_hat, observer.bias_hat
    rec["ep_ret"] = rec["rew"].sum(dim=0)
    if plan is None:
        rec["metrics"] = metrics(rec["eta"], ref, rec["thrust"], rec["angles"], env.dt)
    else:
        rec["metrics"] = metrics(rec["eta"] - rec["setpoint"], torch.zeros(3, n, **f), rec["thrust"], rec["angles"], env.dt)
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
