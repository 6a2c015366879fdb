"""GPU checks of the passive nonlinear DP observer (ml4ca_observer_step, csrc/observer.cu) against its float64
restatement (tests/observer_oracle.py), its restart / reset semantics, argument checks, CUDA-graph capture with the env
step, the Python surface and one closed-loop check of what it is for.

Tolerances, one step from the same state (fp32 kernel against the float64 recurrence; 20 or 1 sub-steps), relative to
each row's scale: wave states xi^ and pose eta^ <= 2e-5 max(1, |x|), velocity nu^ <= 2e-5 max(1, |nu|), bias
b^ <= 1e-4 max(1, |b|).  All four cases (hull 0 and 1, step_dt 0.2 and 0.01 s) pass these bounds on the B200."""
import ctypes

import numpy as np
import pytest
import torch

import observer_oracle as OO
from oracle import constants as C

pytestmark = pytest.mark.gpu

ERR_INVALID = -1
SEA = dict(sigma=(0.1, 0.1, np.deg2rad(2.0)), peak_frequency=(1.0, 2.0), damping=0.1)
TOL = {"xi": 2e-5, "eta": 2e-5, "nu": 2e-5, "bias": 1e-4}
ROWS = {"xi": slice(0, 6), "eta": OO.ETA, "nu": OO.NU, "bias": OO.BIAS}


def np_(t):
    return t.cpu().numpy()


def random_inputs(rng, n):
    x = np.zeros((15, n))
    x[0:6] = rng.normal(size=(6, n)) * 0.05
    x[OO.ETA] = rng.uniform(-1, 1, (3, n)) * np.array([[6.0], [6.0], [3.0]])
    x[OO.NU] = rng.uniform(-1, 1, (3, n)) * np.array([[0.8], [0.3], [0.3]])
    x[OO.BIAS] = rng.normal(size=(3, n)) * np.array([[10.0], [10.0], [5.0]])
    y = x[OO.ETA] + rng.normal(size=(3, n)) * 0.15
    y[2, ::7] += 2 * np.pi                                      # unwrapped headings: the innovation wraps
    thrust = rng.uniform(-100, 100, (3, n))
    angles = rng.uniform(-np.pi, np.pi, (3, n))
    omega = rng.uniform(1.0, 2.0, n)
    f32 = lambda a: a.astype(np.float32)
    return f32(x), f32(y), f32(thrust), f32(angles), f32(omega)


def dev_(a, d):
    return torch.as_tensor(np.ascontiguousarray(a), device=d)


@pytest.mark.parametrize("hull_model", [0, 1])
@pytest.mark.parametrize("step_dt", [0.2, 0.01])
def test_step_matches_oracle(cuda_device, hull_model, step_dt):
    """One step from the same random state, per-env w_o in [1, 2] (plus a few out-of-range values the kernel clamps), odd n."""
    import ml4ca_b200 as M
    n = 4099
    rng = np.random.default_rng(hull_model * 7 + int(step_dt * 100))
    x, y, th, an, om = random_inputs(rng, n)
    om[:4] = [np.nan, -1.0, 0.0, 50.0]
    ob = M.DPObserver(n, step_dt=step_dt, hull_model=hull_model, device=cuda_device)
    ob.state.copy_(dev_(x, cuda_device))
    ob.omega_o.copy_(dev_(om, cuda_device))
    ob.step(dev_(y, cuda_device), dev_(th, cuda_device), dev_(an, cuda_device))
    got = np_(ob.state).astype(np.float64)
    cfg = OO.ObserverCfg(hull_model, step_dt=float(np.float32(step_dt)))
    want = OO.step(cfg, x.astype(np.float64), y.astype(np.float64), th.astype(np.float64), an.astype(np.float64),
                   om.astype(np.float64))
    for k, rows in ROWS.items():
        rel = np.abs(got[rows] - want[rows]) / np.maximum(1.0, np.abs(want[rows]))
        assert rel.max() <= TOL[k], (k, rel.max())


def test_restart_and_reset_bits(cuda_device):
    """Restart columns and masked reset columns equal the reset values bit for bit; the other columns equal a run
    without the restart / mask bits bit for bit."""
    import ml4ca_b200 as M
    n = 2053
    rng = np.random.default_rng(5)
    x, y, th, an, om = random_inputs(rng, n)
    y_t, th_t, an_t = dev_(y, cuda_device), dev_(th, cuda_device), dev_(an, cuda_device)
    A, B = (M.DPObserver(n, device=cuda_device) for _ in range(2))
    for ob in (A, B):
        ob.state.copy_(dev_(x, cuda_device))
        ob.omega_o.copy_(dev_(om, cuda_device))
    m = torch.as_tensor(rng.random(n) < 0.3, device=cuda_device)
    A.step(y_t, th_t, an_t, restart=m.to(torch.uint8) * 3)            # any non-zero byte (a done-flag byte) restarts
    B.step(y_t, th_t, an_t)
    want = torch.zeros(15, n, device=cuda_device)
    want[6:9] = y_t
    assert torch.equal(A.state[:, m], want[:, m]) and torch.equal(A.state[:, ~m], B.state[:, ~m])
    before = B.state.clone()
    B.reset(y_t, mask=m)
    assert torch.equal(B.state[:, m], want[:, m]) and torch.equal(B.state[:, ~m], before[:, ~m])
    B.reset(y_t)
    assert torch.equal(B.state, want)


def test_bad_arguments(cuda_device):
    from ml4ca_b200 import _lib
    L = _lib.lib()
    n = 8
    buf = torch.zeros(15, n, device=cuda_device)
    y, th, an = (torch.zeros(3, n, device=cuda_device) for _ in range(3))
    om = torch.ones(n, device=cuda_device)
    p = _lib.ptr
    s = _lib.current_stream()
    cfg = _lib.ObserverCfg()
    assert L.ml4ca_observer_cfg_default(0, ctypes.byref(cfg)) == 0
    assert L.ml4ca_observer_cfg_default(2, ctypes.byref(cfg)) == ERR_INVALID and b"hull_model" in L.ml4ca_last_error()

    def step(c, n=n, **ptrs):
        a = dict(y=p(y), th=p(th), an=p(an), om=p(om), st=p(buf))
        a.update(ptrs)
        return L.ml4ca_observer_step(c if c is None else ctypes.byref(c), n, a["y"], a["th"], a["an"], a["om"], None, a["st"], s)
    for field, value, msg in (("notch_damping", 0.1, "notch_damping"), ("notch_damping", 0.05, "notch_damping"),
                              ("wave_damping", 0.0, "wave_damping"), ("wave_damping", 1.0, "wave_damping"),
                              ("cutoff_ratio", 1.0, "cutoff_ratio"), ("bias_time_s", -1.0, "bias_time_s"),
                              ("step_dt", 0.0, "step_dt"), ("step_dt", float("nan"), "finite"), ("hull_model", 3, "hull_model")):
        c = _lib.ObserverCfg()
        L.ml4ca_observer_cfg_default(0, ctypes.byref(c))
        setattr(c, field, value)
        assert step(c) == ERR_INVALID, field
        assert msg.encode() in L.ml4ca_last_error(), (field, L.ml4ca_last_error())
    for gain in ("k3", "k4"):
        c = _lib.ObserverCfg()
        L.ml4ca_observer_cfg_default(1, ctypes.byref(c))
        getattr(c, gain)[1] = -1.0
        assert step(c) == ERR_INVALID and b"k3, k4" in L.ml4ca_last_error()
    assert step(None) == ERR_INVALID and b"cfg is NULL" in L.ml4ca_last_error()
    for k in ("y", "th", "an", "om", "st"):
        assert step(cfg, **{k: None}) == ERR_INVALID and b"required" in L.ml4ca_last_error(), k
    assert step(cfg, n=-1) == ERR_INVALID
    assert L.ml4ca_observer_reset(-1, p(y), None, p(buf), s) == ERR_INVALID
    assert L.ml4ca_observer_reset(n, None, None, p(buf), s) == ERR_INVALID
    assert L.ml4ca_observer_reset(n, p(y), None, None, s) == ERR_INVALID
    launches = _lib.launch_count()
    assert step(cfg, n=0) == 0 and L.ml4ca_observer_reset(0, p(y), None, p(buf), s) == 0
    assert _lib.launch_count() == launches
    with pytest.raises(AssertionError, match="unknown observer gains"):
        import ml4ca_b200 as M
        M.DPObserver(n, device=cuda_device, k5=(1, 2, 3))


def test_graph_capture_with_auto_reset(cuda_device):
    """env.step + observer.step(restart=done) under auto_reset, captured once and replayed, equals eager execution bit for
    bit: env state, done flags and the observer state, through in-kernel restarts, with waves on."""
    import ml4ca_b200 as M
    n, T = 3001, 12
    mk = lambda: M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=cuda_device, seed=4,
                               auto_reset=True, max_ep_len=10)
    envs = [mk(), mk()]
    obs_ = [M.DPObserver.for_env(e) for e in envs]
    bufs = [(torch.empty(9, n, device=cuda_device), torch.empty(n, device=cuda_device),
             torch.empty(n, dtype=torch.uint8, device=cuda_device)) for _ in envs]
    for e, ob in zip(envs, obs_):
        e.set_waves(**SEA)
        e.reset()
        ob.omega_o.copy_(e.get_state()["wave_omega"])
        ob.reset(e.get_state()["eta_measured"])
    act = torch.zeros(7, n, device=cuda_device)

    def body(k):
        e, ob, out = envs[k], obs_[k], bufs[k]
        e.step(act, out=out)
        st = e.get_state()
        ob.step(st["eta_measured"], st["prev_thrust"], st["angles"], restart=out[2])

    g = torch.Generator(device=cuda_device)
    g.manual_seed(1)
    actions = [torch.rand(7, n, device=cuda_device, generator=g) * 2 - 1 for _ in range(T + 1)]
    act.copy_(actions[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                # warm-up of the captured env (mirrored eagerly below)
        body(1)
    torch.cuda.current_stream().wait_stream(side)
    body(0)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body(1)
    restarts = 0
    for t in range(1, T + 1):
        act.copy_(actions[t])
        body(0)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(bufs[0][2], bufs[1][2]) and torch.equal(obs_[0].state, obs_[1].state), t
        restarts += int((bufs[0][2] != 0).sum())
    sA, sB = envs[0].get_state(), envs[1].get_state()
    for k in ("eta", "nu", "ep_len", "wave"):
        assert torch.equal(sA[k], sB[k]), k
    assert restarts > n and torch.isfinite(obs_[0].state).all()


def test_python_surface_and_evaluation_wiring(cuda_device):
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    n, T = 12, 30
    env = M.RevoltFinal(M.StandInHull(hull_model=1), testing=True, extended_state=True, cont_ang=True, num_envs=n,
                        device=cuda_device, max_ep_len=400)
    ob = M.DPObserver.for_env(env, peak_frequency=1.2, cutoff_ratio=1.5, k4=(10.0, 20.0, 30.0))
    assert ob.cfg.hull_model == 1 and abs(ob.cfg.step_dt - 0.2) < 1e-7 and ob.cfg.cutoff_ratio == 1.5
    assert list(ob.cfg.k4) == [10.0, 20.0, 30.0] and ob.state.shape == (15, n) and ob.device == env.device
    assert torch.equal(ob.omega_o, torch.full((n,), 1.2, device=cuda_device))
    d = M.DPObserver(n, device=cuda_device)
    assert abs(d.cfg.k4[0] - OO.OBS_K4_PER_MASS * C.M11) < 1e-4 and abs(d.cfg.k3[2] - OO.OBS_K3_PER_K4 * OO.OBS_K4_PER_MASS * C.M33) < 1e-4
    y = torch.randn(3, n, device=cuda_device)
    ob.reset(y)
    st = ob.get_state()
    assert set(st) == {"eta", "nu", "bias", "wave"} and torch.equal(st["eta"], y) and (st["bias"] == 0).all()
    e_hat, n_hat, b_hat = ob.step(y, torch.full((3, n), 50.0, device=cuda_device), torch.zeros(3, n, device=cuda_device))
    assert e_hat.shape == n_hat.shape == b_hat.shape == (3, n) and float(n_hat[0].min()) > 0     # surge thrust: u^ > 0
    assert e_hat.data_ptr() == ob.state[6:9].data_ptr()
    def fresh():                        # every reset draws new waves: repeated runs need an env in the same state
        e = M.RevoltFinal(M.StandInHull(hull_model=1), testing=True, extended_state=True, cont_ang=True, num_envs=n,
                          device=cuda_device, max_ep_len=400, seed=3)
        e.set_waves(**SEA)
        return e
    base = evaluate.run_allocator(fresh(), "pinv", max_ep_len=T)
    again = evaluate.run_allocator(fresh(), "pinv", max_ep_len=T, observer=None)
    assert "eta_hat" not in base and all(torch.equal(base[k], again[k]) for k in base)
    e = fresh()
    rec = evaluate.run_allocator(e, "pinv", max_ep_len=T, observer=M.DPObserver.for_env(e))
    assert rec["eta_hat"].shape == rec["bias_hat"].shape == (T + 1, 3, n) and torch.isfinite(rec["metrics"]).all()
    assert set(base) | {"eta_hat", "bias_hat"} == set(rec)
    from conftest import golden
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=golden("policy_final_80x3.npz")["params"], device=cuda_device)
    for integrator in (False, True):
        r0 = evaluate.run_RL_policy(fresh(), ac, max_ep_len=T, integrator=integrator)
        r1 = evaluate.run_RL_policy(fresh(), ac, max_ep_len=T, integrator=integrator)
        assert "eta_hat" not in r0 and all(torch.equal(r0[k], r1[k]) for k in r0)
        e = fresh()
        r = evaluate.run_RL_policy(e, ac, max_ep_len=T, integrator=integrator, observer=M.DPObserver.for_env(e))
        assert r["eta_hat"].shape == r["bias_hat"].shape == (T + 1, 3, n) and torch.isfinite(r["metrics"]).all()
        assert set(r0) | {"eta_hat", "bias_hat"} == set(r)


# PID + pseudoinverse at sigma_pos = 0.1 m, the 48 runs of tools/observer_eval.py (b) (6 poses x 8 wave seeds, env seed 11),
# 400 steps.  W* with the observer at the fixed w_o = 1.5 rad/s must fall below W_MARGIN x W* without it.  The B200 measured
# 499 J against 1324 J, a ratio of 0.38 (profiles/observer_r3.md (b)); 0.8 leaves room for the fp32 differences of another
# build while still failing if the observer stops filtering the waves.
W_MARGIN = 0.8


def test_observer_lowers_propeller_energy_in_waves(cuda_device):
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    n = 48

    def run(observer):
        env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=cuda_device,
                            max_ep_len=800, seed=11)
        env.set_waves(sigma=(0.1, 0.1, np.deg2rad(2.0)), peak_frequency=(1.0, 2.0), damping=0.1)
        return evaluate.run_allocator(env, "pinv", max_ep_len=400, observer=M.DPObserver.for_env(env) if observer else None)
    w_plain = float(run(False)["metrics"][1].mean())
    w_obs = float(run(True)["metrics"][1].mean())
    assert w_obs < W_MARGIN * w_plain, (w_obs, w_plain)
