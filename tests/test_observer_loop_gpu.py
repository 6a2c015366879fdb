"""GPU checks of the DP observer in the loop (ml4ca_env_set_observer, the OBSV variants of the env-step kernel): twin
equality with a separately stepped observer in every env class and variant, the float64 restatements composed, the cut
and restart semantics, explicit resets and observe(), CUDA graphs, the host-buffer path, detaching and bad arguments,
the evaluation harness and training.

Tolerances.  Without waves the twin's observer sees the same fp32 pose as the fused kernel, and every comparison is bit
for bit.  In waves the twin's measurement y is computed in torch (``measured_pose``) and the kernel's in registers; the
two differ in the last bits of the pose, so the twin's estimates and rows 0-5 are compared within 2e-5 max(1, |x|)
there (the same one-step bound ``test_observer_gpu.py`` states against float64).  Against the float64 restatements the
bounds are those of ``test_observer_gpu.py`` (observer rows) and ``test_waves_gpu.py`` (env rows, observation 5e-5)."""
import ctypes

import numpy as np
import pytest
import torch

import disturbance_oracle as DO
import observer_oracle as OO
import wave_oracle as WO
from oracle import env_oracle as EO

pytestmark = pytest.mark.gpu

ERR_INVALID = -1
DT = float(np.float32(0.2))
SEA = dict(sigma=(0.1, 0.1, np.deg2rad(2.0)), peak_frequency=(1.0, 2.0), damping=0.1)
DIST = dict(current_speed=(0.0, 0.15), current_direction=(0.0, 2 * np.pi), bias_std=(10.0, 10.0, 5.0), bias_time_s=4.0)
WAVE_TOL = 2e-5
OBS_TOL = {"xi": 2e-5, "eta": 2e-5, "nu": 2e-5, "bias": 1e-4}     # test_observer_gpu.py
OBS_ROWS = {"xi": slice(0, 6), "eta": OO.ETA, "nu": OO.NU, "bias": OO.BIAS}

# the nine env classes: (class, cont_ang, extended_state)
CLASSES = [("full", False, False), ("full", False, True), ("simple", False, False), ("limited", False, False),
           ("limited", False, True), ("final", False, False), ("final", False, True), ("final", True, False),
           ("final", True, True)]
VARIANTS = [(lag, dist, wave) for lag in (False, True) for dist in (False, True) for wave in (False, True)]


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


def sensed(st):
    return (st["eta_measured"], st["nu_measured"]) if "eta_measured" in st else (st["eta"], st["nu"])


def error_frame(eta, ref):
    from ml4ca_b200.env import ErrorFrame
    return ErrorFrame(eta.contiguous(), ref, device=eta.device).get_pose()


def rel_close(a, b, tol):
    a, b = a.double(), b.double()
    return float(((a - b).abs() / b.abs().clamp(min=1.0)).max()) <= tol


STATE_KEYS = ("eta", "nu", "prev_thrust", "angles", "ep_len", "current", "bias", "wave", "wave_rate", "wave_omega")


@pytest.mark.parametrize("lag,dist,wave", VARIANTS)
@pytest.mark.parametrize("kind,cont,ext", CLASSES)
def test_twin_equality(cuda_device, kind, cont, ext, lag, dist, wave):
    """An env with an attached observer against a twin without one, whose observer is stepped separately on
    get_state()'s measured pose, prev_thrust and angles: same vessel, reward, flags and rows 6-8; rows 0-5 are the
    separate observer's error frame and velocity.  auto_reset=False: no restarts.

    The OBSV kernel and the kernel the twin runs are compiled separately, and outside the correctly rounded (_rn)
    operations the compiler may form multiply-adds differently in each.  On the B200 build that happens in one case, the
    extended-state DIST kernels without waves, where the reward differs in the last bits: there the reward and the env
    state are compared within 2e-6 max(1, |x|) (as test_disturbance_gpu.py does), everything else bit for bit."""
    import ml4ca_b200 as M
    n, T = 1031, 12
    A, B = (make_env(n, kind, cont, ext, lag, seed=7, max_ep_len=800, device=cuda_device) for _ in range(2))
    for e in (A, B):
        if dist:
            e.set_disturbance(**DIST)
        if wave:
            e.set_waves(**SEA)
        e.reset()
    oA, oB = M.DPObserver.for_env(A), M.DPObserver.for_env(B)
    A.set_observer(oA)
    oB.state.copy_(oA.state)                                     # the same start: eta^ = the measured pose
    g = torch.Generator(device=cuda_device)
    g.manual_seed(3)
    for t in range(T):
        a = torch.rand(A.num_actions, n, device=cuda_device, generator=g) * 2.4 - 1.2
        obA, rA, _, iA = A.step(a)
        obB, rB, _, iB = B.step(a)
        sA, sB = A.get_state(), B.get_state()
        oB.step(sensed(sB)[0], sB["prev_thrust"], sB["angles"])
        assert torch.equal(iA["flags"], iB["flags"]), t
        same = torch.equal if not (dist and ext and not wave) else (lambda x, y: rel_close(x, y, 2e-6))
        assert same(rA, rB), (t, float((rA - rB).abs().max()))
        for k in STATE_KEYS:
            if k in sB:
                assert same(sA[k], sB[k]) if k != "ep_len" else torch.equal(sA[k], sB[k]), (t, k)
        assert torch.equal(obA[6:], obB[6:]), t
        head = torch.cat([error_frame(oB.eta_hat, B._ref), oB.nu_hat])
        if wave:
            assert rel_close(oA.state, oB.state, WAVE_TOL), t
            assert rel_close(obA[0:6], head, WAVE_TOL), t
        else:
            assert torch.equal(oA.state, oB.state), (t, float((oA.state - oB.state).abs().max()))
            assert torch.equal(obA[0:6], head), (t, float((obA[0:6] - head).abs().max()))


@pytest.mark.parametrize("hull_model,lag", [(0, 0.0), (1, 0.92)])
def test_against_float64(cuda_device, hull_model, lag):
    """One step at a time against the float64 restatements composed (env, disturbance, waves, observer), RevoltFinal
    with lag, disturbance and waves; the oracle's observer starts every step from the kernel's observer state."""
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
    ob = M.DPObserver.for_env(env)
    env.set_observer(ob)
    cfg = OO.ObserverCfg(hull_model, step_dt=DT)
    sg = env.get_state()
    for t in range(8):
        for k in ("wave", "wave_rate", "wave_omega", "current", "bias"):
            st[k] = np_(sg[k]).astype(np.float64)
        x0 = np_(ob.state).astype(np.float64)
        a = rng.uniform(-1.0, 1.0, (7, n)).astype(np.float32)
        o64, r64, d64, info = WO.step(spec, st, a.astype(np.float64), waves, dist=dO, seed=seed)
        o, r, d, inf = env.step(torch.as_tensor(a, device=cuda_device))
        sg = env.get_state()
        y64, _ = WO.measured(st['eta'], st['nu'], st['wave'], st['wave_rate'])
        x64 = OO.step(cfg, x0, y64, st['prev_thrust'], st['angles'], np_(ob.omega_o).astype(np.float64))
        x = np_(ob.state).astype(np.float64)
        for k, rows in OBS_ROWS.items():
            rel = np.abs(x[rows] - x64[rows]) / np.maximum(1.0, np.abs(x64[rows]))
            assert rel.max() <= OBS_TOL[k], (t, k, rel.max())
        want = EO.observe(spec, x64[OO.ETA], x64[OO.NU], st['ref'], st['prev_thrust'])
        np.testing.assert_allclose(np_(o)[0:6], want[0:6], rtol=0, atol=1e-4)
        np.testing.assert_allclose(np_(o)[6:9], o64[6:9], rtol=0, atol=5e-5)
        np.testing.assert_allclose(np_(r)[~d64], r64[~d64], rtol=0, atol=2e-4)     # the reward stays the measured one
        np.testing.assert_allclose(np_(sg['eta']), st['eta'], rtol=0, atol=2e-5)
        np.testing.assert_allclose(np_(sg['nu']), st['nu'], rtol=0, atol=2e-6)
        st['eta'], st['nu'] = np_(sg['eta']).astype(np.float64), np_(sg['nu']).astype(np.float64)


def fresh_column(y):
    x = torch.zeros(15, y.shape[1], device=y.device)
    x[6:9] = y
    return x


def test_cut_and_restart(cuda_device):
    """auto_reset over several episodes: cut_obs at an episode-length cut equals bit for bit what an auto_reset=False twin
    with an attached observer returns at that step; at every restart (cut or terminal) the observer column is a fresh
    reset on the new episode's pose and the returned observation has nu^ = 0."""
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib
    n, L = 2048, 10
    A = make_env(n, seed=5, auto_reset=True, max_ep_len=L, device=cuda_device)
    B = make_env(n, seed=5, auto_reset=False, max_ep_len=L, device=cuda_device)
    obs_ = [M.DPObserver.for_env(e) for e in (A, B)]
    for e, ob in zip((A, B), obs_):
        e.reset()
        e.set_observer(ob)
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
            assert torch.equal(obs_[0].state[:, m], fresh_column(st["eta"])[:, m]), t
            assert (oA[3:6, m] == 0).all()
            assert torch.equal(oA[0:3, m], error_frame(st["eta"], A._ref)[:, m])
            restarts += int(m.sum())
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(A._handle, None), "ml4ca_env_set_cut_obs")
    assert cuts > n // 2 and restarts > 2 * n


def test_explicit_resets_and_observe(cuda_device):
    """Masked reset() and reset_to re-initialise only the masked observer columns from the measured pose (waves on); the
    returned rows 3-5 of those columns are 0.  observe() returns the last step's rows 0-5."""
    import ml4ca_b200 as M
    n = 1500
    env = make_env(n, ext=False, seed=8, device=cuda_device)
    env.set_waves(**SEA)
    env.reset()
    ob = M.DPObserver.for_env(env)
    env.set_observer(ob)
    a = torch.full((7, n), 0.3, device=cuda_device)
    for _ in range(4):
        o, _, _, _ = env.step(a)
    assert torch.equal(env.observe(), o)
    mask = torch.zeros(n, dtype=torch.bool)
    mask[::3] = True
    m = mask.to(cuda_device)
    for how in ("sample", "reset_to"):
        before = ob.state.clone()
        if how == "sample":
            o = env.reset(mask=mask)
        else:
            o = env.reset(mask=mask, **{'Hull.PosNED': [1.0, -2.0], 'Hull.PosAttitude': [0, 0, 0.1]})
        st = env.get_state()
        want = fresh_column(st["eta_measured"])
        assert torch.equal(ob.state[:, ~m], before[:, ~m])
        assert torch.equal(ob.state[[0, 1, 2, 3, 4, 5, 9, 10, 11, 12, 13, 14]][:, m], want[[0, 1, 2, 3, 4, 5, 9, 10, 11, 12, 13, 14]][:, m])
        assert rel_close(ob.state[6:9, m], want[6:9, m], WAVE_TOL)
        assert (o[3:6, m] == 0).all()
        assert torch.equal(env.observe()[:, m], o[:, m])
        for _ in range(2):
            o, _, _, _ = env.step(a)
        assert torch.equal(env.observe(), o)


def test_graph_rollout_attach_detach_and_host_path(cuda_device):
    """rollout(graph=True) with an attached observer equals the eager rollout bit for bit; attaching and detaching give
    new graph-cache entries; step_host at 4100 envs equals the device-buffer step bit for bit."""
    import ml4ca_b200 as M
    n, T = 3000, 10
    ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=cuda_device, seed=21)
    envs = [make_env(n, seed=9, auto_reset=True, max_ep_len=12, device=cuda_device) for _ in range(2)]
    bufs = [M.TrajectoryBuffer(9, 7, T, n, device=cuda_device) for _ in range(2)]
    obs_ = [M.DPObserver.for_env(e) for e in envs]
    for e, ob in zip(envs, obs_):
        e.set_waves(**SEA)
        e.reset()
        e.set_observer(ob)
    epoch = 0

    def both(k):
        nonlocal epoch
        for _ in range(k):
            M.rollout(envs[0], ac, bufs[0], seed=5, start_step=epoch * T)
            M.rollout(envs[1], ac, bufs[1], seed=5, start_step=epoch * T, graph=True)
            for name in ("obs_buf", "act_buf", "rew_buf", "logp_buf", "done_buf", "cut_obs"):
                assert torch.equal(getattr(bufs[0], name), getattr(bufs[1], name)), (epoch, name)
            assert torch.equal(obs_[0].state, obs_[1].state), epoch
            epoch += 1
    both(3)
    assert len(bufs[1]._rollout_graphs) == 1
    assert all(e["graph"] is not None for e in bufs[1]._rollout_graphs.values())
    for e in envs:
        e.set_observer(None)
    both(2)
    assert len(bufs[1]._rollout_graphs) == 2
    obs2 = [M.DPObserver.for_env(e) for e in envs]
    for e, ob in zip(envs, obs2):
        e.set_observer(ob)
    both(2)
    assert len(bufs[1]._rollout_graphs) == 3 and torch.equal(obs2[0].state, obs2[1].state)

    n = 4100
    kw = dict(seed=11, auto_reset=True, max_ep_len=12, device=cuda_device)
    A, B = make_env(n, **kw), make_env(n, **kw)
    oA, oB = M.DPObserver.for_env(A), M.DPObserver.for_env(B)
    for e, ob in ((A, oA), (B, oB)):
        e.set_waves(**SEA)
        e.reset()
        e.set_observer(ob)
    g = torch.Generator()
    g.manual_seed(n)
    h_obs, h_rew, h_done = torch.empty(9, n).pin_memory(), torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    for t in range(8):
        h_act = (torch.rand(7, n, generator=g) * 2.4 - 1.2).pin_memory()
        A.step_host(h_act, h_obs, h_rew, h_done)
        o, r, d, info = B.step(h_act.to(cuda_device))
        torch.cuda.synchronize()
        assert torch.equal(h_obs, o.cpu()) and torch.equal(h_rew, r.cpu()) and torch.equal(h_done, info['flags'].cpu()), t
        assert torch.equal(oA.state, oB.state), t


def test_host_path_chunks_advance_the_observer_rows(cuda_device):
    """step_host with chunks smaller than the batch (ML4CA_HOST_CHUNK is read once per process, so the chunk count comes
    from the batch size here: 1 Mi + 4100 envs span two chunks at the default) equals the device-buffer step."""
    import ml4ca_b200 as M
    n = (1 << 20) + 4100
    kw = dict(seed=13, auto_reset=True, max_ep_len=8, device=cuda_device)
    A, B = make_env(n, **kw), make_env(n, **kw)
    oA, oB = M.DPObserver.for_env(A), M.DPObserver.for_env(B)
    for e, ob in ((A, oA), (B, oB)):
        e.reset()
        e.set_observer(ob)
    h_obs, h_rew, h_done = torch.empty(9, n).pin_memory(), torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    g = torch.Generator()
    g.manual_seed(1)
    for t in range(3):
        h_act = (torch.rand(7, n, generator=g) * 2.4 - 1.2).pin_memory()
        A.step_host(h_act, h_obs, h_rew, h_done)
        o, _, _, _ = B.step(h_act.to(cuda_device))
        torch.cuda.synchronize()
        assert torch.equal(h_obs, o.cpu()) and torch.equal(oA.state, oB.state), t


def test_detach_and_bad_arguments(cuda_device):
    """After detaching, the env steps bit-identically to an env that never had an observer; a step_dt mismatch, NULL
    state or omega_o, a wrong num_envs or device are rejected with a message."""
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib
    n = 777
    A, B = (make_env(n, seed=4, device=cuda_device) for _ in range(2))
    for e in (A, B):
        e.set_waves(**SEA)
        e.reset()
    ob = M.DPObserver.for_env(A)
    A.set_observer(ob)
    a = torch.full((7, n), 0.2, device=cuda_device)
    for _ in range(3):
        A.step(a), B.step(a)
    A.set_observer(None)
    assert A._observer is None
    frozen = ob.state.clone()
    for _ in range(3):
        oA, rA, _, iA = A.step(a)
        oB, rB, _, iB = B.step(a)
        assert torch.equal(oA, oB) and torch.equal(rA, rB) and torch.equal(iA["flags"], iB["flags"])
    assert torch.equal(ob.state, frozen)                          # a detached observer is left alone
    with pytest.raises(_lib.Ml4caError, match="step_dt"):
        A.set_observer(M.DPObserver(n, step_dt=0.1, device=cuda_device))
    with pytest.raises(AssertionError, match="envs"):
        A.set_observer(M.DPObserver(n + 1, device=cuda_device))
    with pytest.raises(AssertionError, match="lives on"):
        A.set_observer(M.DPObserver(n, device="cpu"))
    L, s = _lib.lib(), _lib.current_stream()
    good = M.DPObserver.for_env(A)
    for st, om in ((None, _lib.ptr(good.omega_o)), (_lib.ptr(good.state), None)):
        assert L.ml4ca_env_set_observer(A._handle, ctypes.byref(good.cfg), st, om, s) == ERR_INVALID
        assert b"required" in L.ml4ca_last_error()
    bad = _lib.ObserverCfg()
    L.ml4ca_observer_cfg_default(0, ctypes.byref(bad))
    bad.step_dt = DT
    bad.cutoff_ratio = 1.0
    assert L.ml4ca_env_set_observer(A._handle, ctypes.byref(bad), _lib.ptr(good.state), _lib.ptr(good.omega_o), s) == ERR_INVALID
    assert b"cutoff_ratio" in L.ml4ca_last_error()
    assert L.ml4ca_env_set_observer(None, None, None, None, s) == ERR_INVALID
    oA, _, _, _ = A.step(a)                                       # the rejected attachments left the env detached
    oB, _, _, _ = B.step(a)
    assert torch.equal(oA, oB)
    A.set_observer(M.DPObserver.for_env(A, hull_model=1))         # a model-mismatch observer is allowed


def test_evaluation_on_an_attached_env(cuda_device):
    """run_RL_policy (with and without the integrator) and run_allocator on an env with an attached observer match the
    separate-observer path on a plain twin.  In waves the twin's measurement comes from torch: the closed loop carries
    that fp32 difference, so the records agree within 1e-3 (metrics 1e-3 relative) over 40 steps.  A second observer
    raises."""
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    from conftest import golden
    n, T = 24, 40

    def fresh():
        e = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=cuda_device,
                          max_ep_len=400, seed=3)
        e.set_waves(**SEA)
        return e
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=golden("policy_final_80x3.npz")["params"], device=cuda_device)
    runs = [lambda e, **kw: evaluate.run_RL_policy(e, ac, max_ep_len=T, integrator=False, **kw),
            lambda e, **kw: evaluate.run_RL_policy(e, ac, max_ep_len=T, integrator=True, **kw),
            lambda e, **kw: evaluate.run_allocator(e, "pinv", max_ep_len=T, **kw)]
    for run in runs:
        plain = fresh()
        want = run(plain, observer=M.DPObserver.for_env(plain))
        env = fresh()
        env.set_observer(M.DPObserver.for_env(env))
        got = run(env)
        assert set(got) == set(want)
        for k in ("eta", "eta_hat", "bias_hat", "thrust"):
            assert float((got[k] - want[k]).abs().max()) < 1e-3 * max(1.0, float(want[k].abs().max())), k
        assert torch.allclose(got["metrics"], want["metrics"], rtol=1e-3, atol=1e-3)
        with pytest.raises(ValueError, match="attached"):
            run(env, observer=M.DPObserver.for_env(env))
        run(env, observer=env._observer)                          # the attached observer itself is accepted


def test_ppo_learns_with_the_observer_in_the_loop(cuda_device):
    """ppo() at the reference batch (4 envs x 400 steps) in waves (sigma = 0.1 m, 0.1 m, 2 deg) with an attached observer
    learns: from the first epoch's -0.26 reward per step and VVals -0.2 it climbs well above zero.  Measured on the B200
    (three runs): last-10-epoch mean reward per step 0.12-0.25, VVals 7.7-23, EpLen 56-68 after 200 epochs (in waves the
    64 x 64 policy is still far from the calm-water plateau of test_ppo_learns_station_keeping_at_the_reference_batch_size
    at this point).  Loose thresholds: fp32 atomics make runs differ."""
    import ml4ca_b200 as M
    env = make_env(4, seed=0, auto_reset=True, device=cuda_device)
    env.set_waves(**SEA)
    env.reset()
    env.set_observer(M.DPObserver.for_env(env))
    ac, hist = M.ppo(env, steps_per_epoch=400, epochs=200, seed=0)
    first, last = hist[0], hist[-10:]
    assert -0.6 < first["AverageStepReward"] < 0.1 and abs(first["AverageVVals"]) < 5
    assert np.mean([h["AverageStepReward"] for h in last]) > 0.0
    assert np.mean([h["AverageVVals"] for h in last]) > 2.5
    assert np.mean([h["EpLen"] for h in last if h["Episodes"] > 0]) > 35


def test_trpo_tensor_core_graph_with_the_observer(cuda_device):
    """trpo(..., kernel='tensor_core', graph=True): two graph-replayed epochs with an attached observer, finite
    statistics."""
    import ml4ca_b200 as M
    env = make_env(64, seed=2, auto_reset=True, device=cuda_device)
    env.set_waves(**SEA)
    env.reset()
    ob = M.DPObserver.for_env(env)
    env.set_observer(ob)
    ac, hist = M.trpo(env, steps_per_epoch=100, epochs=3, seed=1, graph=True, kernel='tensor_core',
                      hidden_sizes=(80, 80, 80))
    assert len(hist) == 3 and all(np.isfinite(h["AverageStepReward"]) for h in hist)
    assert torch.isfinite(ob.state).all()
