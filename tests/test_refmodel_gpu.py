"""The DP reference model on the device: refmodel_step_kernel and refmodel_reset_kernel against the float64
restatement (tests/refmodel_oracle.py), the bad arguments, the PID's velocity feed-forward (ml4ca_pinv_pid_ff), the
evaluation harness with set-point schedules against loops written out from its primitives, and one closed loop over the
box test against the float64 closed loop."""
import ctypes

import numpy as np
import pytest
import torch

import refmodel_oracle as R
from conftest import golden
from oracle import constants as C
from oracle import eval_oracle as EV
from oracle import pinv_oracle as PO

pytestmark = pytest.mark.gpu


def start_batch(n, seed):
    """Per-env states and set-points: states inside the limits, set-points up to 20 m away (so both limits are hit), and
    every third env with its filter heading and its set-point heading on either side of +-pi."""
    rng = np.random.default_rng(seed)
    x = np.zeros((9, n))
    x[0:2] = rng.uniform(-5, 5, (2, n))
    x[2] = rng.uniform(-np.pi, np.pi, n)
    x[3:6] = rng.uniform(-1, 1, (3, n)) * np.asarray(R.REF_V_MAX)[:, None]
    x[6:9] = rng.uniform(-1, 1, (3, n)) * np.asarray(R.REF_A_MAX)[:, None]
    r = np.zeros((3, n))
    r[0:2] = x[0:2] + rng.uniform(-20, 20, (2, n))
    r[2] = rng.uniform(-np.pi, np.pi, n)
    far = np.arange(n) % 3 == 1
    side = np.where(rng.random(n) < 0.5, 1.0, -1.0)
    x[2, far] = side[far] * (np.pi - rng.uniform(0, 0.4, far.sum()))
    r[2, far] = -side[far] * (np.pi - rng.uniform(0, 0.4, far.sum()))
    return x.astype(np.float32), r.astype(np.float32)


def rows(buf_len, offset, dev):
    """A flat float32 buffer whose data starts ``offset`` floats in (offset 1: 4-byte aligned only)."""
    return torch.zeros(buf_len + offset, dtype=torch.float32, device=dev)[offset:]


def cfg_of(step_dt):
    from ml4ca_b200 import _lib
    cfg = _lib.RefModelCfg()
    assert _lib.lib().ml4ca_refmodel_cfg_default(ctypes.byref(cfg)) == 0
    cfg.step_dt = step_dt
    return cfg


# fp32 rounding alone: the filter is stable, so each sub-step's rounding (~6e-8 relative) decays; over 50 env steps the
# error stays a few ulps of the largest pose (~25 m) -- 2e-4 m leaves room for the clamp and wrap decisions taken
# on values a rounding apart, and is far below any modelling error (e.g. v and a updated in the other order: > 1e-2).
TOL = {"eta": 2e-4, "vel": 2e-5, "acc": 2e-5}


@pytest.mark.parametrize("step_dt", [0.2, 0.01])
@pytest.mark.parametrize("n,offset", [(2 * 256 * 3 + 2, 0), (2 * 256 * 3 + 2, 1), (777, 0), (1, 0)])
def test_step_matches_oracle(cuda_device, step_dt, n, offset):
    """Even and odd n, rows only 4-byte aligned (offset 1), a partial last block, a single env."""
    from ml4ca_b200 import _lib
    x0, r = start_batch(n, seed=n + offset)
    state = rows(9 * n, offset, cuda_device)
    sp = rows(3 * n, offset, cuda_device)
    state.copy_(torch.as_tensor(x0.reshape(-1), device=cuda_device))
    sp.copy_(torch.as_tensor(r.reshape(-1), device=cuda_device))
    cfg = cfg_of(step_dt)
    ocfg = R.RefCfg(step_dt=step_dt)
    want = x0.astype(np.float64)
    for _ in range(50):
        assert _lib.lib().ml4ca_refmodel_step(ctypes.byref(cfg), n, _lib.ptr(sp), _lib.ptr(state), _lib.current_stream()) == 0
        want = R.step(ocfg, want, r.astype(np.float64))
    got = state.view(9, n).cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(got[R.ETA], want[R.ETA], rtol=0, atol=TOL["eta"])
    np.testing.assert_allclose(got[R.VEL], want[R.VEL], rtol=0, atol=TOL["vel"])
    np.testing.assert_allclose(got[R.ACC], want[R.ACC], rtol=0, atol=TOL["acc"])
    assert (np.abs(got[R.VEL]) <= np.asarray(R.REF_V_MAX, dtype=np.float32)[:, None]).all()
    if step_dt == 0.2 and n > 1:                      # 50 x 0.2 s of 20 m steps: both limits reached by some env
        assert (np.abs(got[R.VEL]) == np.asarray(R.REF_V_MAX, dtype=np.float32)[:, None]).any(axis=1).all()


def test_reset_and_python_surface(cuda_device):
    import ml4ca_b200 as M
    n = 1001
    m = M.ReferenceModel(n, device=cuda_device)
    m.state.fill_(7.0)
    eta0 = torch.randn(3, n, device=cuda_device)
    m.reset(eta0)
    assert torch.equal(m.eta_d, eta0) and torch.equal(m.v_d, torch.zeros_like(eta0)) and torch.equal(m.a_d, m.v_d)
    m.reset([1.0, 2.0, 3.0])
    assert torch.equal(m.eta_d, torch.tensor([[1.0], [2.0], [3.0]], device=cuda_device).expand(3, n))
    eta_d, v_d = m.step([1.0, 3.0, 3.0])
    want = R.step(R.RefCfg(), R.reset(np.array([1.0, 2.0, 3.0])), np.array([1.0, 3.0, 3.0]))
    np.testing.assert_allclose(m.state[:, 0].cpu().numpy(), want[:, 0], atol=1e-6)
    assert eta_d.data_ptr() == m.state.data_ptr() and v_d.data_ptr() == m.state[3].data_ptr()
    m2 = M.ReferenceModel(4, step_dt=0.1, device=cuda_device, omega=(0.3, 0.3, 0.3), v_max=(1, 1, 1))
    assert abs(m2.step_dt - 0.1) < 1e-7 and abs(m2.cfg.omega[0] - 0.3) < 1e-7 and m2.cfg.a_max[0] == np.float32(0.05)
    with pytest.raises(AssertionError):
        M.ReferenceModel(4, device=cuda_device, gain=(1, 1, 1))


def test_bad_arguments(cuda_device):
    from ml4ca_b200 import _lib
    L = _lib.lib()
    n = 64
    state, sp, eta0 = (torch.zeros(k, n, device=cuda_device) for k in (9, 3, 3))
    cfg = cfg_of(0.2)
    s = _lib.current_stream()
    before = _lib.launch_count()
    assert L.ml4ca_refmodel_step(ctypes.byref(cfg), 0, _lib.ptr(sp), _lib.ptr(state), s) == 0
    assert L.ml4ca_refmodel_reset(0, _lib.ptr(eta0), _lib.ptr(state), s) == 0
    assert _lib.launch_count() == before                                         # n = 0 launches nothing
    assert L.ml4ca_refmodel_step(None, n, _lib.ptr(sp), _lib.ptr(state), s) == -1
    assert L.ml4ca_refmodel_step(ctypes.byref(cfg), n, None, _lib.ptr(state), s) == -1
    assert L.ml4ca_refmodel_step(ctypes.byref(cfg), n, _lib.ptr(sp), None, s) == -1
    assert L.ml4ca_refmodel_step(ctypes.byref(cfg), -1, _lib.ptr(sp), _lib.ptr(state), s) == -1
    assert L.ml4ca_refmodel_reset(n, None, _lib.ptr(state), s) == -1
    assert L.ml4ca_refmodel_reset(n, _lib.ptr(eta0), None, s) == -1
    assert L.ml4ca_refmodel_cfg_default(None) == -1
    for field, d, value in (("step_dt", None, 0.0), ("step_dt", None, float("nan")), ("zeta", 1, 0.0), ("omega", 2, -0.1),
                            ("omega", 0, float("inf")), ("v_max", 0, 0.0), ("a_max", 2, -1.0),
                            ("omega", 1, 200.0)):              # omega = 200 rad/s at h = 0.01 s: unstable sub-step map
        bad = cfg_of(0.2)
        if d is None:
            setattr(bad, field, value)
        else:
            getattr(bad, field)[d] = value
        assert L.ml4ca_refmodel_step(ctypes.byref(bad), n, _lib.ptr(sp), _lib.ptr(state), s) == -1, (field, value)
        assert L.ml4ca_last_error()
    assert not R.jury_stable(1.0, 200.0, 0.01) and R.jury_stable(1.0, 20.0, 0.01)
    ok = cfg_of(0.2)
    ok.omega[1] = 20.0
    assert L.ml4ca_refmodel_step(ctypes.byref(ok), n, _lib.ptr(sp), _lib.ptr(state), s) == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("n", [5, 4096])
def test_pinv_pid_ff(cuda_device, n):
    """Against float64; and with v_d = 0 bit-equal to ml4ca_pinv_pid (n even: the two-envs-per-thread path, odd: scalar)."""
    import ml4ca_b200 as M
    eta, nu, _, _ = PO.synth_batch(n, seed=4)
    rng = np.random.default_rng(5)
    ref = (rng.uniform(-1, 1, (3, n)) * np.array([[4.0], [4.0], [0.6]])).astype(np.float32)
    vd = (rng.uniform(-1, 1, (3, n)) * np.array([[0.3], [0.3], [0.2]])).astype(np.float32)
    eta, nu = eta.astype(np.float32), nu.astype(np.float32)
    t = lambda a: torch.as_tensor(a, device=cuda_device)
    integ = torch.zeros(3, n, device=cuda_device)
    want_i = np.zeros((3, n))
    for _ in range(2):
        n_pct, alpha, tau = M.pinv_pid(t(eta), t(nu), t(ref), integ, return_tau=True, nu_d=t(vd))
        wtau, want_i = R.pid_ff(eta.astype(np.float64), nu.astype(np.float64), ref.astype(np.float64), vd.astype(np.float64),
                                want_i)
        np.testing.assert_allclose(tau.cpu().numpy(), wtau, rtol=2e-6, atol=2e-4)
        np.testing.assert_allclose(integ.cpu().numpy(), want_i, rtol=1e-6, atol=1e-6)
        wn, wa = PO.allocate(tau.cpu().numpy().astype(np.float64))
        K = np.asarray(C.K_THRUST)[:, None]
        got = n_pct.cpu().numpy().astype(np.float64)
        np.testing.assert_allclose(K * got * np.abs(got), K * wn * np.abs(wn), rtol=1e-5, atol=5e-5)
    # the feed-forward changes the wrench where the PID is not saturated
    plain = PO.pid(eta.astype(np.float64), nu.astype(np.float64), ref.astype(np.float64), np.zeros((3, n)))[0]
    ff = R.pid_ff(eta.astype(np.float64), nu.astype(np.float64), ref.astype(np.float64), vd.astype(np.float64),
                  np.zeros((3, n)))[0]
    assert np.abs(plain - ff).max() > 1.0
    i1, i2 = torch.zeros(3, n, device=cuda_device), torch.zeros(3, n, device=cuda_device)
    a = M.pinv_pid(t(eta), t(nu), t(ref), i1, return_tau=True)
    b = M.pinv_pid(t(eta), t(nu), t(ref), i2, return_tau=True, nu_d=torch.zeros(3, n, device=cuda_device))
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert torch.equal(i1, i2)


# ---- evaluation harness ------------------------------------------------------------------------------------------------

N, T = 12, 40


def small_schedule(dev):
    """Per-env set-points, changing at steps 7 and 19, some with a heading across +-pi from the last."""
    rng = np.random.default_rng(8)
    sp = (rng.uniform(-1, 1, (3, 3, N)) * np.array([[2.0], [2.0], [0.4]])).astype(np.float32)
    sp[2, 2, ::4] = np.float32(3.0)
    sp[1, 2, ::4] = np.float32(-3.0)
    return np.array([0, 7, 19]), torch.as_tensor(sp, device=dev)


def make_env(M, dev):
    return M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=N, device=dev)


def s_of(steps, sp, t):
    return sp[int(np.searchsorted(steps, t, side="right")) - 1]


def reset_at(env, s0):
    eta0 = s0.double().cpu().numpy()
    env.set_ref(s0)
    return env.reset(**{'Hull.PosNED': eta0[0:2], 'Hull.PosAttitude': np.stack([np.zeros(N), np.zeros(N), eta0[2]]),
                        'Hull.VelocityNu': np.zeros((6, N))})


def check_common(rec, want, steps, sp, dt, with_model):
    for key, val in want.items():
        assert torch.equal(rec[key], torch.stack(val)), key
    s = torch.stack([s_of(steps, sp, t) for t in range(T + 1)])
    assert torch.equal(rec["setpoint"], s)
    if not with_model:
        assert torch.equal(rec["ref"], s)
    eta, sp64 = rec["eta"].cpu().numpy().astype(np.float64), s.cpu().numpy().astype(np.float64)
    iae = [EV.iae(eta[:, :, i], sp64[:, :, i], dt) for i in range(N)]
    np.testing.assert_allclose(rec["metrics"][0].cpu().numpy(), iae, rtol=2e-5)


@pytest.mark.parametrize("with_model", [False, True])
@pytest.mark.parametrize("method", ["pinv", "qp"])
def test_run_allocator_with_schedule_matches_the_primitives(cuda_device, method, with_model):
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib, evaluate
    from ml4ca_b200.qp_allocator import QPTA
    steps, sp = small_schedule(cuda_device)
    env = make_env(M, cuda_device)
    model = M.ReferenceModel.for_env(env) if with_model else None
    rec = evaluate.run_allocator(env, method, max_ep_len=T, schedule=(steps, sp), reference_model=model)

    env = make_env(M, cuda_device)
    model = M.ReferenceModel.for_env(env) if with_model else None
    f = dict(dtype=torch.float32, device=cuda_device)
    reset_at(env, s_of(steps, sp, 0))
    ref, vd = s_of(steps, sp, 0).clone(), torch.zeros(3, N, **f)
    if model is not None:
        model.reset(ref)
    st = env.get_state()
    integ = torch.zeros(3, N, **f)
    qp = QPTA(num_envs=N, device=cuda_device) if method == "qp" else None
    slew, trust = torch.tensor([[4.0], [2.0], [2.0]], **f), torch.ones(N, **f)
    lx, ly = (-1.12, -1.12, 1.08), (-0.15, 0.15, 0.0)
    action = torch.empty(env.num_actions, N, **f)
    want = {"eta": [st["eta"]], "thrust": [torch.zeros(3, N, **f)], "ref": [ref.clone()]}
    if with_model:
        want["v_d"] = [vd.clone()]
    clipped = []
    for t in range(T):
        n_pct, alpha, tau = M.pinv_pid(st["eta"], st["nu"], ref, integ, return_tau=True, nu_d=vd if with_model else None)
        if qp is not None:
            f0, f1, f2, a0, a1 = qp._prev
            c0, s0, c1, s1 = torch.cos(a0), torch.sin(a0), torch.cos(a1), torch.sin(a1)
            now = torch.stack([f0 * c0 + f1 * c1, f0 * s0 + f1 * s1 + f2,
                               f0 * (lx[0] * s0 - ly[0] * c0) + f1 * (lx[1] * s1 - ly[1] * c1) + f2 * lx[2]])
            lim = slew * trust[None, :]
            clipped.append(((tau - now).abs() > lim).any(dim=0))
            qp.tau_controller_callback_func(now + torch.minimum(torch.maximum(tau - now, -lim), lim))
            ok = (qp.last_status & 1).bool()
            trust = torch.where(ok, (trust * 2).clamp(max=1.0), trust * 0.5)
            n_pct, alpha = qp.last_output[0:3].contiguous(), qp.last_output[3:5].contiguous()
        _lib.check(_lib.lib().ml4ca_alloc_to_action(N, 1, float(env.real_action_bounds[3]), _lib.ptr(n_pct), _lib.ptr(alpha),
                                                    _lib.ptr(action), _lib.current_stream()))
        if model is not None:
            model.step(s_of(steps, sp, t))
            ref, vd = model.eta_d.clone(), model.v_d.clone()
            want["v_d"].append(vd)
        else:
            ref = s_of(steps, sp, t + 1).clone()
        env.set_ref(ref)
        env.step(action)
        st = env.get_state()
        want["eta"].append(st["eta"]), want["thrust"].append(st["prev_thrust"]), want["ref"].append(ref)
    check_common(rec, want, steps, sp, float(env.dt), with_model)
    if qp is not None:
        assert torch.equal(rec["demand_clipped"], torch.stack(clipped))


@pytest.mark.parametrize("with_model", [False, True])
@pytest.mark.parametrize("variant", ["plain", "integrator", "observer", "attached"])
def test_run_RL_policy_with_schedule_matches_the_primitives(cuda_device, variant, with_model):
    """The state assembly (integrator, separate observer) must use r(t); an attached observer's observation is formed
    by the env with the reference it was given before the step."""
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib, evaluate
    g = golden("policy_final_80x3.npz")
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=g["params"], device=cuda_device)
    steps, sp = small_schedule(cuda_device)
    integrator = variant == "integrator"

    def make():
        env = make_env(M, cuda_device)
        obs = None
        if variant in ("observer", "attached"):
            obs = M.DPObserver.for_env(env)
            if variant == "attached":
                env.set_observer(obs)
        return env, obs, (M.ReferenceModel.for_env(env) if with_model else None)
    env, obs, model = make()
    rec = evaluate.run_RL_policy(env, ac, max_ep_len=T, integrator=integrator, schedule=(steps, sp), reference_model=model,
                                 observer=obs if variant == "observer" else None)

    env, obs, model = make()
    f = dict(dtype=torch.float32, device=cuda_device)
    o = reset_at(env, s_of(steps, sp, 0))
    ref = s_of(steps, sp, 0).clone()
    if model is not None:
        model.reset(ref)
    st = env.get_state()
    if variant == "observer":
        obs.reset(evaluate.sensed(st)[0])
    integ, t_inside = torch.zeros(3, N, **f), torch.zeros(N, **f)
    prev_u, ros = torch.zeros(6, N, **f), torch.empty(9, N, **f)
    want = {"obs": [o], "eta": [st["eta"]], "thrust": [torch.zeros(3, N, **f)], "ref": [ref.clone()]}
    if with_model:
        want["v_d"] = [torch.zeros(3, N, **f)]
    for t in range(T):
        x = o
        if integrator or variant == "observer":
            eta_s, nu_s = evaluate.sensed(st) if obs is None else (obs.eta_hat.contiguous(), obs.nu_hat.contiguous())
            _lib.check(_lib.lib().ml4ca_ros_state(N, _lib.ptr(eta_s), _lib.ptr(nu_s), _lib.ptr(ref), _lib.ptr(prev_u),
                                                  _lib.ptr(integ if integrator else None),
                                                  _lib.ptr(t_inside if integrator else None), float(env.dt), _lib.ptr(ros),
                                                  _lib.current_stream()))
            x = o.clone()
            x[0:3] = ros[0:3]
            if obs is not None:
                x[3:6] = nu_s
        a = ac.get_action(x)
        if model is not None:
            model.step(s_of(steps, sp, t))
            ref = model.eta_d.clone()
            want["v_d"].append(model.v_d.clone())
        else:
            ref = s_of(steps, sp, t + 1).clone()
        env.set_ref(ref)
        o, _, _, _ = env.step(a)
        st = env.get_state()
        if variant == "observer":
            obs.step(evaluate.sensed(st)[0], st["prev_thrust"], st["angles"])
        want["obs"].append(o), want["eta"].append(st["eta"]), want["thrust"].append(st["prev_thrust"])
        want["ref"].append(ref)
    check_common(rec, want, steps, sp, float(env.dt), with_model)
    if not with_model:                             # a schedule change at step k first shows in sample k
        k = int(steps[1])
        assert not torch.equal(rec["ref"][k], rec["ref"][k - 1])
    for s in (7, 19, T):                           # each observation is the error frame of its own reference
        if variant != "attached":
            ef = M.ErrorFrame(rec["eta"][s], rec["ref"][s], device=cuda_device).get_pose()
            np.testing.assert_allclose(rec["obs"][s][0:3].cpu().numpy(), ef.cpu().numpy(), rtol=0, atol=1e-5)


def test_harness_errors_on_the_device(cuda_device):
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    env = make_env(M, cuda_device)
    steps, sp = small_schedule(cuda_device)
    with pytest.raises(ValueError):
        evaluate.run_allocator(env, "pinv", schedule=(steps, sp), reference_model=M.ReferenceModel(N + 1, device=cuda_device))
    with pytest.raises(ValueError):
        evaluate.run_allocator(env, "pinv", schedule=(steps, sp),
                               reference_model=M.ReferenceModel(N, step_dt=0.1, device=cuda_device))
    with pytest.raises(ValueError):
        evaluate.run_RL_policy(env, None, schedule=(steps, sp), new_ref=sp[1], ref_change_at=3)
    with pytest.raises(ValueError):
        evaluate.run_allocator(env, "pinv", schedule=(steps[::-1].copy(), sp))


def test_box_test_closed_loop_matches_float64(cuda_device):
    """PID + feed-forward + pseudoinverse with the reference model over the whole box test in calm water, against the
    float64 closed loop.  The loop is stable, so fp32 and float64 stay within a few millimetres and a tenth of a degree."""
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    steps, sp = evaluate.box_test_schedule()
    n = 4
    env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=cuda_device,
                        max_ep_len=4000)
    rec = evaluate.run_allocator(env, "pinv", schedule=(steps, sp), reference_model=M.ReferenceModel.for_env(env))
    want = R.closed_loop(steps, sp, int(steps[-1]), R.RefCfg())
    eta = rec["eta"].cpu().numpy().astype(np.float64)
    for i in range(n):
        np.testing.assert_allclose(eta[:, 0:2, i], want["eta"][:, 0:2], rtol=0, atol=2e-2)
        np.testing.assert_allclose(eta[:, 2, i], want["eta"][:, 2], rtol=0, atol=np.deg2rad(0.2))
        np.testing.assert_allclose(rec["ref"][:, :, i].cpu().numpy(), want["ref"], rtol=0, atol=2e-4)
    iae = EV.iae(want["eta"], want["setpoint"], 0.2)
    np.testing.assert_allclose(rec["metrics"][0].cpu().numpy(), iae, rtol=2e-3)
