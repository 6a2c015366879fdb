"""GPU checks of the DP reference model in the loop (ml4ca_env_set_refmodel, the REF variants of the env-step kernel):
twin equality with a separately stepped reference model in every env class and variant, with and without an attached
observer; the float64 restatements composed; the cut and restart semantics; explicit resets, attach and observe(); CUDA
graphs and the host-buffer path; detaching and bad arguments; the evaluation harness and training.

The twin is an env without the model whose set-point is the separate model's eta_d: ``ReferenceModel.step(s)``, then
``set_ref(eta_d.clone())``, then ``step``.  The in-loop step is declared to equal that sequence bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

import disturbance_oracle as DO
import observer_oracle as OO
import refmodel_oracle as RO
import wave_oracle as WO
from oracle import env_oracle as EO

pytestmark = pytest.mark.gpu

ERR_INVALID = -1
DT = float(np.float32(0.2))
SEA = dict(sigma=(0.1, 0.1, np.deg2rad(2.0)), peak_frequency=(1.0, 2.0), damping=0.1)
DIST = dict(current_speed=(0.0, 0.15), current_direction=(0.0, 2 * np.pi), bias_std=(10.0, 10.0, 5.0), bias_time_s=4.0)
WAVE_TOL = 2e-5                                                   # test_observer_loop_gpu.py
OBS_TOL = {"xi": 2e-5, "eta": 2e-5, "nu": 2e-5, "bias": 1e-4}     # test_observer_gpu.py
OBS_ROWS = {"xi": slice(0, 6), "eta": OO.ETA, "nu": OO.NU, "bias": OO.BIAS}

CLASSES = [("full", False, False), ("full", False, True), ("simple", False, False), ("limited", False, False),
           ("limited", False, True), ("final", False, False), ("final", False, True), ("final", True, False),
           ("final", True, True)]
VARIANTS = [(lag, dist, wave) for lag in (False, True) for dist in (False, True) for wave in (False, True)]
STATE_KEYS = ("eta", "nu", "prev_thrust", "angles", "ep_len", "current", "bias", "wave", "wave_rate", "wave_omega")


def np_(t):
    return t.cpu().numpy()


def make_env(n, kind="final", cont=True, ext=True, lag=False, **kw):
    import ml4ca_b200.env as E
    hull = E.StandInHull(hull_model=1 if lag else 0)            # model 1 carries the 0.92 s wrench lag
    cls = {"full": E.Revolt, "simple": E.RevoltSimple, "limited": E.RevoltLimited, "final": E.RevoltFinal}[kind]
    if kind == "final":
        return cls(hull, extended_state=ext, cont_ang=cont, num_envs=n, **kw)
    if kind == "full":
        return cls(digitwin=hull, extended_state=ext, num_envs=n, **kw)
    return cls(hull, extended_state=ext, num_envs=n, **kw)


def setpoints(n, seed, dev, scale=(3.0, 3.0, 0.5)):
    """Per-env set-points; every fifth env has its heading set-point near +-pi (the model's wrapped heading error)."""
    rng = np.random.default_rng(seed)
    s = rng.uniform(-1, 1, (3, n)) * np.asarray(scale)[:, None]
    far = np.arange(n) % 5 == 2
    s[2, far] = np.where(rng.random(far.sum()) < 0.5, 1.0, -1.0) * (np.pi - 0.05)
    return torch.as_tensor(s, dtype=torch.float32, device=dev)


def error_frame(eta, ref):
    from ml4ca_b200.env import ErrorFrame
    return ErrorFrame(eta.contiguous(), ref.contiguous(), device=eta.device).get_pose()


def rel_close(a, b, tol):
    a, b = a.double(), b.double()
    return float(((a - b).abs() / b.abs().clamp(min=1.0)).max()) <= tol


def fresh_column(eta):
    x = torch.zeros(9, eta.shape[1], device=eta.device)
    x[0:3] = eta
    return x


@pytest.mark.parametrize("obsv", [False, True])
@pytest.mark.parametrize("lag,dist,wave", VARIANTS)
@pytest.mark.parametrize("kind,cont,ext", CLASSES)
def test_twin_equality(cuda_device, kind, cont, ext, lag, dist, wave, obsv):
    """An env with an attached model against a twin that is driven by a separate ReferenceModel (step(s), set_ref(eta_d),
    step): observation, reward, flags, every state row and the model state, bit for bit over 20 steps.  Per-env
    set-points that change at step 10; auto_reset=False.  With ``obsv`` both envs carry an attached observer."""
    import ml4ca_b200 as M
    n, T = 1031, 20
    A, B = (make_env(n, kind, cont, ext, lag, seed=7, max_ep_len=800, device=cuda_device) for _ in range(2))
    for e in (A, B):
        if dist:
            e.set_disturbance(**DIST)
        if wave:
            e.set_waves(**SEA)
        e.reset()
    if obsv:
        oA, oB = M.DPObserver.for_env(A), M.DPObserver.for_env(B)
        A.set_observer(oA)
        B.set_observer(oB)
    mA, mB = M.ReferenceModel.for_env(A), M.ReferenceModel.for_env(B)
    A.set_reference_model(mA)
    mB.reset(B.get_state()["eta"])
    assert torch.equal(mA.state, mB.state)
    s = setpoints(n, 1, cuda_device)
    A.set_ref(s)
    g = torch.Generator(device=cuda_device)
    g.manual_seed(3)
    for t in range(T):
        if t == 10:
            s = setpoints(n, 2, cuda_device)
            A.set_ref(s)
        a = torch.rand(A.num_actions, n, device=cuda_device, generator=g) * 2.4 - 1.2
        mB.step(s)
        B.set_ref(mB.eta_d.clone())
        obA, rA, _, iA = A.step(a)
        obB, rB, _, iB = B.step(a)
        sA, sB = A.get_state(), B.get_state()
        assert torch.equal(iA["flags"], iB["flags"]), t
        assert torch.equal(rA, rB), (t, float((rA - rB).abs().max()))
        assert torch.equal(obA, obB), (t, float((obA - obB).abs().max()))
        for k in STATE_KEYS:
            if k in sB:
                assert torch.equal(sA[k], sB[k]), (t, k)
        assert torch.equal(mA.state, mB.state), (t, float((mA.state - mB.state).abs().max()))
        if obsv:
            assert torch.equal(oA.state, oB.state), t
    assert torch.equal(A._ref, s)                                 # the set-point rows keep the operator's command


@pytest.mark.parametrize("hull_model,lag,obsv", [(0, 0.0, False), (1, 0.92, True)])
def test_against_float64(cuda_device, hull_model, lag, obsv):
    """One step at a time against the float64 restatements composed (reference model, env, disturbance, waves and, with
    ``obsv``, the observer), RevoltFinal with disturbance and waves: the model steps from the kernel's model state on s,
    and the env step is formed against the float64 eta_d."""
    import ml4ca_b200 as M
    import ml4ca_b200.env as E
    n, seed = 2053, 12
    spec = EO.EnvSpec('final', True, True, max_ep_len=800, hull_model=hull_model, actuator_lag_s=lag)
    waves = WO.Waves(step_dt=DT, **SEA)
    dO = DO.Disturbance(step_dt=DT, **DIST)
    env = E.RevoltFinal(E.StandInHull(hull_model=hull_model, actuator_lag_s=lag), extended_state=True, cont_ang=True,
                        num_envs=n, seed=seed, device=cuda_device)
    env.set_disturbance(**DIST)
    env.set_waves(**SEA)
    rng = np.random.default_rng(hull_model)
    eta0 = (rng.uniform(-1, 1, (3, n)) * np.array([[4.0], [4.0], [0.4]])).astype(np.float32).astype(np.float64)
    nu0 = (rng.uniform(-1, 1, (3, n)) * np.array([[0.5], [0.1], [0.2]])).astype(np.float32).astype(np.float64)
    st = EO.new_state(spec, n)
    WO.reset(spec, st, waves, dist=dO, eta=eta0, nu=nu0, seed=seed)
    z = 0 * eta0[0]
    env.reset(**{'Hull.PosNED': eta0[:2], 'Hull.PosAttitude': np.stack([z, z, eta0[2]]),
                 'Hull.VelocityNu': np.stack([nu0[0], nu0[1], z, z, z, nu0[2]])})
    s = setpoints(n, 5, cuda_device)
    env.set_ref(s)
    s64 = np_(s).astype(np.float64)
    if obsv:
        ob = M.DPObserver.for_env(env)
        env.set_observer(ob)
        ocfg = OO.ObserverCfg(hull_model, step_dt=DT)
    m = M.ReferenceModel.for_env(env)
    env.set_reference_model(m)
    np.testing.assert_array_equal(np_(m.state), RO.reset(eta0))
    rcfg = RO.RefCfg(step_dt=DT)
    sg = env.get_state()
    for t in range(8):
        for k in ("wave", "wave_rate", "wave_omega", "current", "bias"):
            st[k] = np_(sg[k]).astype(np.float64)
        r64 = RO.step(rcfg, np_(m.state).astype(np.float64), s64)
        st['ref'] = r64[RO.ETA]
        if obsv:
            x0 = np_(ob.state).astype(np.float64)
        a = rng.uniform(-1.0, 1.0, (7, n)).astype(np.float32)
        o64, r_64, d64, _ = WO.step(spec, st, a.astype(np.float64), waves, dist=dO, seed=seed)
        o, r, d, _ = env.step(torch.as_tensor(a, device=cuda_device))
        sg = env.get_state()
        x = np_(m.state).astype(np.float64)
        np.testing.assert_allclose(x[RO.ETA], r64[RO.ETA], rtol=0, atol=2e-5)
        np.testing.assert_allclose(x[RO.VEL], r64[RO.VEL], rtol=0, atol=2e-6)
        np.testing.assert_allclose(x[RO.ACC], r64[RO.ACC], rtol=0, atol=2e-6)
        if obsv:
            y64, _ = WO.measured(st['eta'], st['nu'], st['wave'], st['wave_rate'])
            xo64 = OO.step(ocfg, x0, y64, st['prev_thrust'], st['angles'], np_(ob.omega_o).astype(np.float64))
            xo = np_(ob.state).astype(np.float64)
            for k, rows in OBS_ROWS.items():
                rel = np.abs(xo[rows] - xo64[rows]) / np.maximum(1.0, np.abs(xo64[rows]))
                assert rel.max() <= OBS_TOL[k], (t, k, rel.max())
            want = EO.observe(spec, xo64[OO.ETA], xo64[OO.NU], r64[RO.ETA], st['prev_thrust'])
            np.testing.assert_allclose(np_(o)[0:6], want[0:6], rtol=0, atol=1e-4)
        else:
            np.testing.assert_allclose(np_(o)[0:6], o64[0:6], rtol=0, atol=5e-5)
        np.testing.assert_allclose(np_(o)[6:9], o64[6:9], rtol=0, atol=5e-5)
        np.testing.assert_allclose(np_(r)[~d64], r_64[~d64], rtol=0, atol=2e-4)     # the reward against eta_d
        assert np.array_equal(np_(d).astype(bool), d64)
        np.testing.assert_allclose(np_(sg['eta']), st['eta'], rtol=0, atol=2e-5)
        np.testing.assert_allclose(np_(sg['nu']), st['nu'], rtol=0, atol=2e-6)
        st['eta'], st['nu'] = np_(sg['eta']).astype(np.float64), np_(sg['nu']).astype(np.float64)


@pytest.mark.parametrize("wave", [False, True])
def test_cut_and_restart(cuda_device, wave):
    """auto_reset over several episodes with per-env set-points: cut_obs at an episode-length cut equals bit for bit what
    an auto_reset=False twin with an attached model returns at that step; at every restart (cut or terminal) the model
    column is (eta, 0, 0) of the new episode's LF pose, and the returned rows 0-2 are exactly 0 in calm water and the
    error of the wave motion in waves."""
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib
    n, L = 2048, 10
    A = make_env(n, seed=5, auto_reset=True, max_ep_len=L, device=cuda_device)
    B = make_env(n, seed=5, auto_reset=False, max_ep_len=L, device=cuda_device)
    models = [M.ReferenceModel.for_env(e) for e in (A, B)]
    s = setpoints(n, 3, cuda_device)
    for e, m in zip((A, B), models):
        if wave:
            e.set_waves(**SEA)
        e.reset()
        e.set_ref(s)
        e.set_reference_model(m)
    cut = torch.full((9, n), float('nan'), device=cuda_device)
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(A._handle, _lib.ptr(cut)), "ml4ca_env_set_cut_obs")
    g = torch.Generator(device=cuda_device)
    g.manual_seed(2)
    twin_ok = torch.ones(n, dtype=torch.bool, device=cuda_device)
    restarts = cuts = 0
    for t in range(3 * A.max_ep_len):
        a = torch.rand(7, n, device=cuda_device, generator=g) * 2.4 - 1.2
        oA, _, _, iA = A.step(a)
        oB, _, _, iB = B.step(a)
        f = iA["flags"]
        if t < A.max_ep_len:
            twin_ok &= iA["flags"] == iB["flags"]
            if t < A.max_ep_len - 1:
                twin_ok &= f == 0
            else:
                at_cut = twin_ok & (f == 2)
                assert float(at_cut.float().mean()) > 0.5
                assert torch.equal(cut[:, at_cut], oB[:, at_cut])
                assert not torch.equal(oA[:, at_cut], oB[:, at_cut])
                cuts += int(at_cut.sum())
        m = f != 0
        if m.any():
            st = A.get_state()
            assert torch.equal(models[0].state[:, m], fresh_column(st["eta"])[:, m]), t
            if wave:
                assert rel_close(oA[0:3, m], error_frame(st["eta_measured"], st["eta"])[:, m], WAVE_TOL), t
                assert (oA[0:3, m] != 0).any()
            else:
                assert (oA[0:3, m] == 0).all(), t
            restarts += int(m.sum())
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(A._handle, None), "ml4ca_env_set_cut_obs")
    assert cuts > n // 2 and restarts > 2 * n
    assert torch.equal(A._ref, s)


@pytest.mark.parametrize("wave", [False, True])
def test_explicit_resets_attach_and_observe(cuda_device, wave):
    """Masked reset() and reset_to start only the masked model columns again at the LF pose; the returned rows 0-2 of those
    columns are exactly 0 in calm water (the wave motion's error in waves).  An unmasked reset and attaching start every
    column at the LF pose, and attaching updates rows 0-2 of the last observation.  observe() forms rows 0-2 against
    eta_d."""
    import ml4ca_b200 as M
    n = 1500
    env = make_env(n, ext=False, seed=8, device=cuda_device)
    if wave:
        env.set_waves(**SEA)
    env.reset()
    env.set_ref(setpoints(n, 4, cuda_device))
    m = M.ReferenceModel.for_env(env)
    a = torch.full((7, n), 0.3, device=cuda_device)
    env.step(a)
    env.set_reference_model(m)
    st = env.get_state()
    assert torch.equal(m.state, fresh_column(st["eta"]))
    pose = st.get("eta_measured", st["eta"])
    assert torch.equal(env._obs[0:3], error_frame(pose, st["eta"]))
    for _ in range(4):
        o, _, _, _ = env.step(a)
    assert torch.equal(env.observe(), o)
    assert (m.v_d != 0).any()
    mask = torch.zeros(n, dtype=torch.bool)
    mask[::3] = True
    k = mask.to(cuda_device)

    def check_fresh(o, cols):
        st = env.get_state()
        assert torch.equal(m.state[:, cols], fresh_column(st["eta"])[:, cols])
        if wave:
            assert rel_close(o[0:3, cols], error_frame(st["eta_measured"], st["eta"])[:, cols], WAVE_TOL)
        else:
            assert (o[0:3, cols] == 0).all()
        assert torch.equal(env.observe()[:, cols], o[:, cols])

    for how in ("sample", "reset_to"):
        before = m.state.clone()
        if how == "sample":
            o = env.reset(mask=mask)
        else:
            o = env.reset(mask=mask, **{'Hull.PosNED': [1.0, -2.0], 'Hull.PosAttitude': [0, 0, 0.1]})
        assert torch.equal(m.state[:, ~k], before[:, ~k])
        check_fresh(o, k)
        for _ in range(2):
            o, _, _, _ = env.step(a)
        assert torch.equal(env.observe(), o)
    o = env.reset()
    check_fresh(o, torch.ones(n, dtype=torch.bool, device=cuda_device))


def test_graph_rollout_attach_detach_and_host_path(cuda_device):
    """rollout(graph=True) with an attached model equals the eager rollout bit for bit; attaching, detaching and attaching a
    model of another configuration give new graph-cache entries; step_host at 4100 envs equals the device-buffer step."""
    import ml4ca_b200 as M
    n, T = 3000, 10
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=cuda_device, seed=21)
    envs = [make_env(n, seed=9, auto_reset=True, max_ep_len=12, device=cuda_device) for _ in range(2)]
    bufs = [M.TrajectoryBuffer(9, 7, T, n, device=cuda_device) for _ in range(2)]
    models = [M.ReferenceModel.for_env(e) for e in envs]
    s = setpoints(n, 6, cuda_device)
    for e, m in zip(envs, models):
        e.set_waves(**SEA)
        e.reset()
        e.set_ref(s)
        e.set_reference_model(m)
    epoch = 0

    def both(k, ms):
        nonlocal epoch
        for _ in range(k):
            M.rollout(envs[0], ac, bufs[0], seed=5, start_step=epoch * T)
            M.rollout(envs[1], ac, bufs[1], seed=5, start_step=epoch * T, graph=True)
            for name in ("obs_buf", "act_buf", "rew_buf", "logp_buf", "done_buf", "cut_obs"):
                assert torch.equal(getattr(bufs[0], name), getattr(bufs[1], name)), (epoch, name)
            if ms is not None:
                assert torch.equal(ms[0].state, ms[1].state), epoch
            epoch += 1
    both(3, models)
    assert len(bufs[1]._rollout_graphs) == 1
    assert all(e["graph"] is not None for e in bufs[1]._rollout_graphs.values())
    for e in envs:
        e.set_reference_model(None)
    both(2, None)
    assert len(bufs[1]._rollout_graphs) == 2
    models2 = [M.ReferenceModel.for_env(e, omega=(0.3, 0.3, 0.3)) for e in envs]
    for e, m in zip(envs, models2):
        e.set_reference_model(m)
    both(2, models2)
    assert len(bufs[1]._rollout_graphs) == 3

    n = 4100
    kw = dict(seed=11, auto_reset=True, max_ep_len=12, device=cuda_device)
    A, B = make_env(n, **kw), make_env(n, **kw)
    mA, mB = M.ReferenceModel.for_env(A), M.ReferenceModel.for_env(B)
    s = setpoints(n, 7, cuda_device)
    for e, m in ((A, mA), (B, mB)):
        e.set_waves(**SEA)
        e.reset()
        e.set_ref(s)
        e.set_reference_model(m)
    g = torch.Generator()
    g.manual_seed(n)
    h_obs, h_rew, h_done = torch.empty(9, n).pin_memory(), torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    for t in range(8):
        h_act = (torch.rand(7, n, generator=g) * 2.4 - 1.2).pin_memory()
        A.step_host(h_act, h_obs, h_rew, h_done)
        o, r, d, info = B.step(h_act.to(cuda_device))
        torch.cuda.synchronize()
        assert torch.equal(h_obs, o.cpu()) and torch.equal(h_rew, r.cpu()) and torch.equal(h_done, info['flags'].cpu()), t
        assert torch.equal(mA.state, mB.state), t


def test_host_path_chunks_advance_the_model_rows(cuda_device):
    """step_host over two pipeline chunks (1 Mi + 4100 envs at the default chunk) equals the device-buffer step, model
    state included: each chunk advances its own rows of the model state."""
    import ml4ca_b200 as M
    n = (1 << 20) + 4100
    kw = dict(seed=13, auto_reset=True, max_ep_len=8, device=cuda_device)
    A, B = make_env(n, **kw), make_env(n, **kw)
    mA, mB = M.ReferenceModel.for_env(A), M.ReferenceModel.for_env(B)
    s = setpoints(n, 8, cuda_device)
    for e, m in ((A, mA), (B, mB)):
        e.reset()
        e.set_ref(s)
        e.set_reference_model(m)
    h_obs, h_rew, h_done = torch.empty(9, n).pin_memory(), torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    g = torch.Generator()
    g.manual_seed(1)
    for t in range(3):
        h_act = (torch.rand(7, n, generator=g) * 2.4 - 1.2).pin_memory()
        A.step_host(h_act, h_obs, h_rew, h_done)
        o, _, _, _ = B.step(h_act.to(cuda_device))
        torch.cuda.synchronize()
        assert torch.equal(h_obs, o.cpu()) and torch.equal(mA.state, mB.state), t


def test_detach_and_bad_arguments(cuda_device):
    """After detaching, the env steps bit-identically to an env that never had a model, and the detached model is left
    alone; a wrong num_envs, device or step_dt, a NULL state and a configuration that fails the Jury test are rejected."""
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib
    n = 777
    A, B = (make_env(n, seed=4, device=cuda_device) for _ in range(2))
    s = setpoints(n, 9, cuda_device)
    for e in (A, B):
        e.set_waves(**SEA)
        e.reset()
        e.set_ref(s)
    m = M.ReferenceModel.for_env(A)
    A.set_reference_model(m)
    a = torch.full((7, n), 0.2, device=cuda_device)
    for _ in range(3):
        A.step(a), B.step(a)
    A.set_reference_model(None)
    assert A._refmodel is None
    frozen = m.state.clone()
    for _ in range(3):
        oA, rA, _, iA = A.step(a)
        oB, rB, _, iB = B.step(a)
        assert torch.equal(oA, oB) and torch.equal(rA, rB) and torch.equal(iA["flags"], iB["flags"])
    assert torch.equal(m.state, frozen)
    with pytest.raises(_lib.Ml4caError, match="step_dt"):
        A.set_reference_model(M.ReferenceModel(n, step_dt=0.1, device=cuda_device))
    with pytest.raises(AssertionError, match="envs"):
        A.set_reference_model(M.ReferenceModel(n + 1, device=cuda_device))
    with pytest.raises(AssertionError, match="lives on"):
        A.set_reference_model(M.ReferenceModel(n, device="cpu"))
    with pytest.raises(_lib.Ml4caError, match="Jury"):
        A.set_reference_model(M.ReferenceModel.for_env(A, omega=(200.0, 0.2, 0.2)))
    L, st = _lib.lib(), _lib.current_stream()
    good = M.ReferenceModel.for_env(A)
    assert L.ml4ca_env_set_refmodel(A._handle, ctypes.byref(good.cfg), None, st) == ERR_INVALID
    assert b"required" in L.ml4ca_last_error()
    assert L.ml4ca_env_set_refmodel(None, None, None, st) == ERR_INVALID
    assert A._refmodel is None
    oA, _, _, _ = A.step(a)                                       # the rejected attachments left the env detached
    oB, _, _, _ = B.step(a)
    assert torch.equal(oA, oB)


def test_evaluation_on_an_attached_env(cuda_device):
    """run_allocator (pinv, qp) and run_RL_policy (plain, integrator, attached observer) on the box-test schedule, on an env
    with the model attached, against the same call with reference_model= on a plain env: every record and the metrics
    identical.  A second model raises ValueError.  Without a schedule the attached model guides the fixed-test-pose runs
    to the env's set-point, scored against it."""
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    from conftest import golden
    n = 24
    sched = evaluate.box_test_schedule(hold_s=8.0)                # the box test with 40-step legs: 240 steps

    def fresh(observer=False):
        e = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=cuda_device,
                          max_ep_len=400, seed=3)
        if observer:
            e.set_observer(M.DPObserver.for_env(e))
        return e
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=golden("policy_final_80x3.npz")["params"], device=cuda_device)
    runs = [(lambda e, **kw: evaluate.run_allocator(e, "pinv", schedule=sched, **kw), False),
            (lambda e, **kw: evaluate.run_allocator(e, "qp", schedule=sched, **kw), False),
            (lambda e, **kw: evaluate.run_RL_policy(e, ac, schedule=sched, **kw), False),
            (lambda e, **kw: evaluate.run_RL_policy(e, ac, schedule=sched, integrator=True, **kw), False),
            (lambda e, **kw: evaluate.run_RL_policy(e, ac, schedule=sched, **kw), True)]
    for run, observer in runs:
        plain = fresh(observer)
        want = run(plain, reference_model=M.ReferenceModel.for_env(plain))
        env = fresh(observer)
        env.set_reference_model(M.ReferenceModel.for_env(env))
        got = run(env)
        assert set(got) == set(want)
        for k in want:
            assert torch.equal(got[k], want[k]), k
        with pytest.raises(ValueError, match="attached"):
            run(env, reference_model=M.ReferenceModel.for_env(env))
        run(env, reference_model=env._refmodel)                  # the attached model itself is accepted

    env = fresh()
    env.set_ref(torch.tensor([1.0, -1.0, 0.2], device=cuda_device))
    env.set_reference_model(M.ReferenceModel.for_env(env))
    T = 60
    for rec in (evaluate.run_allocator(env, "pinv", max_ep_len=T), evaluate.run_RL_policy(env, ac, max_ep_len=T)):
        eta0 = torch.as_tensor(evaluate.fixed_test_poses(n), dtype=torch.float32, device=cuda_device)
        assert torch.equal(rec["ref"][0], eta0) and torch.equal(rec["v_d"][0], torch.zeros_like(eta0))
        assert torch.equal(rec["setpoint"], env._ref[None].expand(T + 1, 3, n))
        assert (rec["v_d"][1:].abs().amax(dim=(0, 2)) > 0).all()
        want = evaluate.metrics(rec["eta"] - rec["setpoint"], torch.zeros(3, n, device=cuda_device), rec["thrust"],
                                rec["angles"], env.dt)
        assert torch.equal(rec["metrics"], want)
    with pytest.raises(ValueError, match="replaces"):
        evaluate.run_RL_policy(env, ac, max_ep_len=T, new_ref=[0, 0, 0], ref_change_at=5)


def test_ppo_learns_with_the_reference_model_in_the_loop(cuda_device):
    """ppo() at the reference batch (4 envs x 400 steps), calm water, with an attached model: every episode is a filtered
    move toward the set-point followed by a hold, and the policy learns it.  Measured on the B200 (one run): first-10-epoch
    reward per step 0.16-0.54 and VVals -4 to 22; after 200 epochs, last 10: reward per step 0.66-2.0, VVals 62-157, EpLen
    400.  Loose thresholds: fp32 atomics make runs differ."""
    import ml4ca_b200 as M
    env = make_env(4, seed=0, auto_reset=True, device=cuda_device)
    env.reset()
    env.set_reference_model(M.ReferenceModel.for_env(env))
    ac, hist = M.ppo(env, steps_per_epoch=400, epochs=200, seed=0)
    first, last = hist[:10], hist[-10:]
    r0 = np.mean([h["AverageStepReward"] for h in first])
    r1 = np.mean([h["AverageStepReward"] for h in last])
    assert r1 > r0 + 0.3
    assert np.mean([h["AverageVVals"] for h in last]) > 25
    assert np.mean([h["EpLen"] for h in last if h["Episodes"] > 0]) > 200


def test_trpo_tensor_core_graph_with_the_model_and_an_observer(cuda_device):
    """trpo(..., kernel='tensor_core', graph=True): three graph-replayed epochs with an attached model and observer, in
    waves, finite statistics."""
    import ml4ca_b200 as M
    env = make_env(64, seed=2, auto_reset=True, device=cuda_device)
    env.set_waves(**SEA)
    env.reset()
    env.set_observer(M.DPObserver.for_env(env))
    m = M.ReferenceModel.for_env(env)
    env.set_reference_model(m)
    ac, hist = M.trpo(env, steps_per_epoch=100, epochs=3, seed=1, graph=True, kernel='tensor_core',
                      hidden_sizes=(80, 80, 80))
    assert len(hist) == 3 and all(np.isfinite(h["AverageStepReward"]) for h in hist)
    assert torch.isfinite(m.state).all()
