"""Evaluation harness (SURVEY.md 8f rank 2): metric kernel against the restated plot-script formulas, and the shipped
80x80x80 checkpoint driven through run_RL_policy from the fixed test poses."""
import os
import sys
import types

import numpy as np
import pytest

from conftest import golden
from oracle import eval_oracle as EV
from oracle import ref_loader


@pytest.mark.skipif(not ref_loader.have_checkout(), reason="reference checkout not present")
def test_iae_oracle_equals_reference_common_py():
    """results/all_plots/common.py IAE itself (matplotlib stubbed out) on a random run."""
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.gridspec"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].gridspec = sys.modules["matplotlib.gridspec"]
    sys.modules["matplotlib.pyplot"].rcParams = {}
    sys.modules["matplotlib"].rcParams = {}
    sys.path.insert(0, os.path.join(ref_loader.REFERENCE_ROOT, "results", "all_plots"))
    try:
        import importlib
        common = importlib.import_module("common")
    finally:
        sys.path.pop(0)
    rng = np.random.default_rng(0)
    T, dt = 50, 0.2
    eta = rng.normal(size=(T, 3)) * np.array([3, 3, 0.4])
    times = np.arange(T) * dt
    const = np.array([0.5, -0.2, 0.1])
    changing = np.tile(const, (T, 1))
    changing[T // 3:] = [-1.5, 2.0, -0.3]                        # a set-point change during the run: one set-point per sample
    for ref in (const, changing):
        r_deg = np.broadcast_to(ref, (T, 3)).copy()
        e_deg = eta.copy()
        e_deg[:, 2], r_deg[:, 2] = np.rad2deg(eta[:, 2]), np.rad2deg(r_deg[:, 2])
        _, cumsum = common.IAE(e_deg / np.array([5., 5., 25.]), r_deg / np.array([5., 5., 25.]), times)
        assert abs(cumsum[-1] - EV.iae(eta, ref, dt)) < 1e-12


@pytest.mark.gpu
def test_metric_kernel_matches_restatement(cuda_device):
    import torch
    from ml4ca_b200 import evaluate
    rng = np.random.default_rng(1)
    T, n, dt = 60, 300, 0.2
    eta = (rng.normal(size=(T, 3, n)) * np.array([3, 3, 0.5])[None, :, None]).astype(np.float32)
    ref = (rng.normal(size=(3, n)) * 0.3).astype(np.float32)
    thrust = rng.uniform(-100, 100, (T, 3, n)).astype(np.float32)
    angles = rng.uniform(-np.pi, np.pi, (T, 2, n)).astype(np.float32)
    dev = lambda x: torch.as_tensor(x, device=cuda_device)
    out = evaluate.metrics(dev(eta), dev(ref), dev(thrust), dev(angles), dt).cpu().numpy()
    for i in range(0, n, 7):
        want = (EV.iae(eta[:, :, i], ref[:, i], dt), EV.work(thrust[:, :, i], dt), EV.iadc(thrust[:, :, i], angles[:, :, i]))
        np.testing.assert_allclose(out[:, i], want, rtol=2e-5)


@pytest.mark.gpu
def test_shipped_policy_from_fixed_test_poses(cuda_device):
    """test_policy.py:97-186 with the shipped final model (80x80x80, leaky-ReLU) in the batched env: every run starts on
    the r = 5 m circle of simtools.py:91-107; the policy was trained in the absent Cybersea simulator, so only
    structural properties are asserted on the stand-in hull."""
    import torch
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    g = golden("policy_final_80x3.npz")
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=g["params"], device=cuda_device)
    n = 12
    env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=cuda_device)
    rec = evaluate.run_RL_policy(env, ac, max_ep_len=100)
    eta0 = rec["eta"][0].cpu().numpy()
    np.testing.assert_allclose(np.hypot(eta0[0], eta0[1]), 5.0, rtol=1e-6)
    np.testing.assert_allclose(eta0, evaluate.fixed_test_poses(n), atol=1e-6)
    assert torch.equal(rec["eta"][:, :, 0:6], rec["eta"][:, :, 6:12])          # deterministic policy: pose k == pose k + 6
    m = rec["metrics"].cpu().numpy()
    assert np.isfinite(m).all() and (m >= 0).all() and (m[0] > 0).all()
    assert rec["thrust"].abs().max() <= 100.0 and rec["ep_ret"].shape == (n,)


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["pinv", "qp"])
def test_classical_allocators_hold_station_in_the_batched_env(cuda_device, method):
    """PID -> allocator -> env, closed loop from the fixed test poses: the vessel must approach the origin (the action
    map inversion, the allocator order port/star/bow vs the env order bow/port/star and the thrust law all have to be
    right for that), and the QP allocator's commands must respect its rate limits."""
    import torch
    import ml4ca_b200 as M
    from ml4ca_b200 import evaluate
    n = 12
    env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=cuda_device)
    rec = evaluate.run_allocator(env, method=method, max_ep_len=300)
    eta = rec["eta"].cpu().numpy()
    d0, d1 = np.hypot(eta[0, 0], eta[0, 1]), np.hypot(eta[-1, 0], eta[-1, 1])
    assert np.allclose(d0, 5.0, rtol=1e-6) and (d1 < 1.5).all(), d1            # 60 s of DP: within 1.5 m of the set-point
    assert (np.abs(eta[-1, 2]) < np.deg2rad(10 if method == 'pinv' else 45)).all()    # the rate-limited QP loop turns slowly
    m = rec["metrics"].cpu().numpy()
    assert np.isfinite(m).all() and (m[0] > 0).all()
    if method == "qp":
        thr = rec["thrust"].cpu().numpy()
        force = np.sign(thr) * thr ** 2 * np.array([0.0009, 0.00205, 0.00205])[None, :, None]      # env order bow, port, star
        dF = np.abs(np.diff(force[1:], axis=0))
        assert (dF[:, 0] <= 2.0 + 1e-2).all() and (dF[:, 1:] <= 5.0 + 1e-2).all()       # qp_allocator.py:57 rate limits


@pytest.mark.gpu
@pytest.mark.parametrize("with_observer", [False, True])
def test_setpoint_change_matches_a_loop_of_the_primitives(cuda_device, with_observer):
    """run_RL_policy(new_ref=..., ref_change_at=k, integrator=True), with and without the DP observer, against the same
    evaluation written out here from its primitives (ac.get_action, ml4ca_ros_state, env.step) with per-env set-points.
    The env takes a new set-point after the step that carries it (customEnv.py:131), so observation s is formed with the
    old set-point up to s = k + 1 and with the new one from s = k + 2; the state assembly of each sample must use that
    sample's set-point, and the IAE must integrate against it sample by sample."""
    import torch
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib, evaluate
    g = golden("policy_final_80x3.npz")
    ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=g["params"], device=cuda_device)
    n, T, k = 12, 40, 8
    rng = np.random.default_rng(3)
    old = (rng.uniform(-1, 1, (3, n)) * np.array([[2.0], [2.0], [0.3]])).astype(np.float32)
    new = (rng.uniform(-1, 1, (3, n)) * np.array([[3.0], [3.0], [0.5]])).astype(np.float32)
    f = dict(dtype=torch.float32, device=cuda_device)

    def make():
        env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=cuda_device)
        env.set_ref(old)
        return env, (M.DPObserver.for_env(env) if with_observer else None)
    env, obs = make()
    rec = evaluate.run_RL_policy(env, ac, max_ep_len=T, new_ref=torch.as_tensor(new, **f), ref_change_at=k, integrator=True,
                                 observer=obs)

    env, obs = make()
    old_t, new_t = torch.as_tensor(old, **f), torch.as_tensor(new, **f)
    ref_of = lambda s: old_t if s <= k + 1 else new_t                          # the set-point observation s is formed with
    eta0 = evaluate.fixed_test_poses(n)
    o = env.reset(**{'Hull.PosNED': eta0[0:2], 'Hull.PosAttitude': np.stack([np.zeros(n), np.zeros(n), eta0[2]]),
                     'Hull.VelocityNu': np.zeros((6, n))})
    st = env.get_state()
    if obs is not None:
        obs.reset(evaluate.sensed(st)[0])
    integ, t_inside = torch.zeros(3, n, **f), torch.zeros(n, **f)
    prev_u, ros = torch.zeros(6, n, **f), torch.empty(9, n, **f)
    want = {"obs": [o], "eta": [st["eta"]], "thrust": [torch.zeros(3, n, **f)]}
    for t in range(T):
        eta_s, nu_s = evaluate.sensed(st) if obs is None else (obs.eta_hat.contiguous(), obs.nu_hat.contiguous())
        _lib.check(_lib.lib().ml4ca_ros_state(n, _lib.ptr(eta_s), _lib.ptr(nu_s), _lib.ptr(ref_of(t)), _lib.ptr(prev_u),
                                              _lib.ptr(integ), _lib.ptr(t_inside), float(env.dt), _lib.ptr(ros),
                                              _lib.current_stream()))
        x = o.clone()
        x[0:3] = ros[0:3]
        if obs is not None:
            x[3:6] = nu_s
        a = ac.get_action(x)
        if t == k:
            o, _, _, _ = env.step(torch.zeros_like(a), new_ref=new_t.clone())
        else:
            o, _, _, _ = env.step(a)
        st = env.get_state()
        if obs is not None:
            obs.step(evaluate.sensed(st)[0], st["prev_thrust"], st["angles"])
        want["obs"].append(o), want["eta"].append(st["eta"]), want["thrust"].append(st["prev_thrust"])
    for key in ("obs", "eta", "thrust"):
        assert torch.equal(rec[key], torch.stack(want[key])), key
    ref = np.stack([ref_of(s).cpu().numpy() for s in range(T + 1)]).astype(np.float64)       # [T + 1, 3, n]
    eta = rec["eta"].cpu().numpy().astype(np.float64)
    iae = [EV.iae(eta[:, :, i], ref[:, :, i], float(env.dt)) for i in range(n)]
    np.testing.assert_allclose(rec["metrics"][0].cpu().numpy(), iae, rtol=2e-5)
    assert not np.allclose(iae, [EV.iae(eta[:, :, i], old[:, i], float(env.dt)) for i in range(n)], rtol=1e-3)
    np.testing.assert_array_equal(rec["ref"].cpu().numpy(), ref.astype(np.float32))
    for s in (k + 1, k + 2, T):                                   # each observation is the error frame of its own set-point
        ef = M.ErrorFrame(rec["eta"][s], rec["ref"][s], device=cuda_device).get_pose()
        np.testing.assert_allclose(rec["obs"][s][0:3].cpu().numpy(), ef.cpu().numpy(), rtol=0, atol=1e-5)
