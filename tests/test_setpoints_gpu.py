"""GPU checks of per-env set-points (ml4ca_env_set_ref) in every compiled env-step kernel, the reset kernel, observe()
and the host-buffer pipeline, against the float64 restatements (oracle/env_oracle.py, tests/disturbance_oracle.py,
tests/wave_oracle.py), whose state carries 'ref'.

Every env gets its own set-point: N, E ~ U(+-4 m), psi ~ U(+-0.6 rad), except every eighth env, whose set-point heading
sits near +pi while its vessel heading starts near -pi: the heading error is then ~ -2 pi and stays unwrapped (the
deg=True quirk of errorFrame.py), so the observation's heading row is far beyond its bound.

The matrix covers the nine env classes that build, each with the default dispatch at an odd n (one env per thread) and at
n % 4 == 0 (two envs per thread), and with the scalar LAG, DIST, DIST + LAG, WAVE, WAVE + LAG, WAVE + DIST and
WAVE + DIST + LAG kernels.  The four-env kernel and the chunked host-buffer pipeline are selected by environment
variables read once per process (ML4CA_ENV_VEC, ML4CA_ENV_THREADS, ML4CA_HOST_CHUNK), so they run in a child process
(this file run as a script) whose records are checked here.

Protocol of tests/test_waves_gpu.py::test_wave_step_matches_oracle: reset_to from seeded poses; 3-step episodes with
auto_reset, so that cuts, terminations and in-kernel restarts occur; after each step the oracle continues from the
kernel's LF state, and the envs the kernel restarted are reset in the oracle from the kernel's new state.  Tolerances
are those of tests/test_env_gpu.py and tests/test_disturbance_gpu.py: observation 2e-5 (5e-5 with waves or the
disturbance), reward 1e-4 (2e-4), position 2e-5, velocity 2e-6; the flags are exact wherever the float64 observation is
clear of its bounds by ten times the observation tolerance."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT  # first: puts the repository root on sys.path when this file runs as the child process
import disturbance_oracle as DO
import wave_oracle as WO
from oracle import env_oracle as EO

pytestmark = pytest.mark.gpu

DT = float(np.float32(0.2))
L = 6                                                     # max_ep_len in the reference's units: 3-step episodes
STEPS = 5
SEA = dict(sigma=(0.1, 0.1, np.deg2rad(2.0)), peak_frequency=(1.0, 2.0), damping=0.1)
DIST = dict(current_speed=(0.0, 0.2), current_direction=(-np.pi, np.pi), bias_std=(15.0, 10.0, 8.0), bias_time_s=4.0)

# (kind, cont_ang, extended_state) of every env class that builds
CLASSES = [('full', False, False), ('full', False, True), ('limited', False, False), ('limited', False, True),
           ('simple', False, False), ('final', False, False), ('final', False, True), ('final', True, False),
           ('final', True, True)]
CLASS_IDS = ['%s-%s-%s' % (k, 'cont' if c else 'wrap', 'ext' if e else 'std') for k, c, e in CLASSES]
# (name, n, lag, disturbance, waves): n odd -> one env per thread, n % 4 == 0 -> two envs per thread (default dispatch)
VARIANTS = [('vec1', 517, False, False, False), ('vec2', 516, False, False, False), ('lag', 517, True, False, False),
            ('dist', 517, False, True, False), ('dist_lag', 517, True, True, False), ('wave', 517, False, False, True),
            ('wave_lag', 517, True, False, True), ('wave_dist', 517, False, True, True),
            ('wave_dist_lag', 517, True, True, True)]
STATE_KEYS = ('eta', 'nu', 'current', 'bias', 'wave', 'wave_rate', 'wave_omega')


def make_env(kind, cont, ext, n, hull_kw=None, **kw):
    import ml4ca_b200.env as E
    hull = E.StandInHull(**(hull_kw or {}))
    if kind == 'full':
        return E.Revolt(digitwin=hull, extended_state=ext, num_envs=n, **kw)
    if kind == 'final':
        return E.RevoltFinal(hull, extended_state=ext, cont_ang=cont, num_envs=n, **kw)
    cls = E.RevoltLimited if kind == 'limited' else E.RevoltSimple
    return cls(hull, extended_state=ext, num_envs=n, **kw)


def init_kw(eta, nu):
    z = 0 * eta[0]
    return {'Hull.PosNED': eta[:2], 'Hull.PosAttitude': np.stack([z, z, eta[2]]),
            'Hull.VelocityNu': np.stack([nu[0], nu[1], z, z, z, nu[2]])}


def setpoints_and_poses(rng, n):
    """Per-env set-points ref [3, n] and start poses eta [3, n], nu [3, n] (float32 values in float64 arrays), and the
    mask of the envs whose set-point heading is near +pi and vessel heading near -pi."""
    ref = rng.uniform(-1, 1, (3, n)) * np.array([[4.0], [4.0], [0.6]])
    eta = rng.uniform(-1, 1, (3, n)) * np.array([[3.0], [3.0], [0.3]])
    nu = rng.uniform(-1, 1, (3, n)) * np.array([[0.5], [0.1], [0.2]])
    far = np.arange(n) % 8 == 3
    ref[2, far] = np.pi - rng.uniform(0, 0.2, far.sum())
    eta[2, far] = -np.pi + rng.uniform(0, 0.2, far.sum())
    f = lambda x: x.astype(np.float32).astype(np.float64)
    return f(ref), f(eta), f(nu), far


def np_(t):
    return t.cpu().numpy()


def kernel_state(env):
    sg = env.get_state()
    return {k: np_(sg[k]).astype(np.float64) for k in STATE_KEYS if k in sg}


def set_cut_obs(env, buf):
    from ml4ca_b200 import _lib
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(env._handle, None if buf is None else _lib.ptr(buf)), "ml4ca_env_set_cut_obs")


def run_kernel(env, rng, steps):
    """Step ``env`` with uniform random actions, the cut observation buffer set; -> records stacked over the steps: a, o,
    r, flags, cut [steps, ...] and the kernel's state (STATE_KEYS) after the reset and after every step [steps + 1, ...]."""
    n = env.num_envs
    rec = {k: [] for k in ('a', 'o', 'r', 'flags', 'cut')}
    states = [kernel_state(env)]
    cut = torch.full((env.num_states, n), float('nan'), device=env.device)
    set_cut_obs(env, cut)
    try:
        for _ in range(steps):
            a = rng.uniform(-1, 1, (env.num_actions, n)).astype(np.float32)
            o, r, _, info = env.step(torch.as_tensor(a, device=env.device))
            for k, v in (('a', a), ('o', np_(o)), ('r', np_(r)), ('flags', np_(info['flags'])), ('cut', np_(cut))):
                rec[k].append(v)
            states.append(kernel_state(env))
    finally:
        set_cut_obs(env, None)
    out = {k: np.stack(v) for k, v in rec.items()}
    for k in states[0]:
        out[k] = np.stack([s[k] for s in states])
    return out


def check_against_oracle(spec, st, rec, waves=None, dist=None, seed=0):
    """Replay the kernel's records ``rec`` (run_kernel) on the oracle state ``st`` (after its reset); -> the number of
    in-kernel restarts and of cut observations checked."""
    noisy = waves is not None or dist is not None
    tol_o, tol_r = (5e-5, 2e-4) if noisy else (2e-5, 1e-4)
    bounds = np.asarray(spec.ss_bounds)[:, None]
    restarts = cuts = 0
    for t in range(rec['a'].shape[0]):
        for k in ('current', 'bias', 'wave', 'wave_rate', 'wave_omega'):
            if k in rec:
                st[k] = rec[k][t].copy()                       # the kernel's disturbance / wave state before the step
        a = rec['a'][t].astype(np.float64)
        if waves is not None:
            o64, r64, d64, info = WO.step(spec, st, a, waves, dist=dist, seed=seed)
        elif dist is not None:
            o64, r64, d64, info = DO.step(spec, st, a, dist, seed=seed)
        else:
            o64, r64, d64, info = EO.step(spec, st, a)
        o, r, flags = rec['o'][t], rec['r'][t], rec['flags'][t]
        eta, nu = rec['eta'][t + 1], rec['nu'][t + 1]
        restarted = flags != 0
        keep = ~restarted
        msg = 'step %d' % t
        np.testing.assert_array_equal((flags >> 1) & 1, info['truncated'].astype(np.uint8), err_msg=msg)
        clear = np.min(np.abs(np.abs(o64[:6]) - bounds), axis=0) > 10 * tol_o
        assert clear.mean() > 0.95, msg
        np.testing.assert_array_equal((flags & 1)[clear], d64[clear].astype(np.uint8), err_msg=msg)
        np.testing.assert_allclose(eta[:, keep], st['eta'][:, keep], rtol=0, atol=2e-5, err_msg=msg)
        np.testing.assert_allclose(nu[:, keep], st['nu'][:, keep], rtol=0, atol=2e-6, err_msg=msg)
        np.testing.assert_allclose(o[:, keep], o64[:, keep], rtol=0, atol=tol_o, err_msg=msg)
        np.testing.assert_allclose(r, r64, rtol=0, atol=tol_r, err_msg=msg)   # the step's reward, restarted or not
        cut_now = flags == 2                                   # cut at the episode length only: the observation it returned
        np.testing.assert_allclose(rec['cut'][t][:, cut_now], o64[:, cut_now], rtol=0, atol=tol_o, err_msg=msg)
        cuts += int(cut_now.sum())
        st['eta'][:, keep], st['nu'][:, keep] = eta[:, keep], nu[:, keep]
        if restarted.any():                                    # the kernel's restart, from the state it drew
            kw = dict(mask=restarted, eta=eta, nu=nu, seed=seed)
            if waves is not None:
                WO.reset(spec, st, waves, dist=dist, **kw)
                for k in ('wave', 'wave_rate', 'wave_omega'):
                    st[k][..., restarted] = rec[k][t + 1][..., restarted]
                o_re = WO.observe(spec, st)
            else:
                if dist is not None:
                    DO.reset(spec, st, dist, **kw)
                else:
                    EO.reset(spec, st, **kw)
                o_re = EO.observe(spec, st['eta'], st['nu'], st['ref'], st['prev_thrust'])
            np.testing.assert_allclose(o[:, restarted], o_re[:, restarted], rtol=0, atol=tol_o, err_msg=msg)
            restarts += int(restarted.sum())
    return restarts, cuts


@pytest.mark.parametrize("variant", VARIANTS, ids=[v[0] for v in VARIANTS])
@pytest.mark.parametrize("cls", CLASSES, ids=CLASS_IDS)
def test_step_with_setpoints_matches_oracle(cuda_device, cls, variant):
    """reset_to, then STEPS steps of every kernel variant of every env class with per-env set-points: the reset and
    restart observations, the step's observation, reward, flags, hull state and the saved cut observation."""
    kind, cont, ext = cls
    name, n, lag, dist, waves = variant
    seed = 17
    hull_kw = dict(hull_model=1, actuator_lag_s=0.92) if lag else dict(hull_model=0, actuator_lag_s=0.0)
    spec = EO.EnvSpec(kind, cont, ext, max_ep_len=L, **hull_kw)
    wO = WO.Waves(step_dt=DT, **SEA) if waves else None
    dO = DO.Disturbance(step_dt=DT, **DIST) if dist else None
    env = make_env(kind, cont, ext, n, hull_kw=hull_kw, max_ep_len=L, auto_reset=True, seed=seed, device=cuda_device)
    if dist:
        env.set_disturbance(**DIST)
    if waves:
        env.set_waves(**SEA)
    rng = np.random.default_rng(CLASSES.index(cls) * 100 + VARIANTS.index(variant))
    ref, eta0, nu0, far = setpoints_and_poses(rng, n)
    env.set_ref(torch.as_tensor(ref, dtype=torch.float32, device=cuda_device))
    st = EO.new_state(spec, n)
    st['ref'] = ref.copy()
    if waves:
        o_ref = WO.reset(spec, st, wO, dist=dO, eta=eta0, nu=nu0, seed=seed)
    elif dist:
        o_ref = DO.reset(spec, st, dO, eta=eta0, nu=nu0, seed=seed)
    else:
        o_ref = EO.reset(spec, st, eta=eta0, nu=nu0)
    o0 = np_(env.reset(**init_kw(eta0, nu0)))
    np.testing.assert_allclose(o0, o_ref, rtol=0, atol=5e-5 if (dist or waves) else 2e-5)
    assert (o0[2, far] < -np.pi).all()                        # unwrapped heading error, beyond every heading bound
    rec = run_kernel(env, rng, STEPS)
    restarts, cuts = check_against_oracle(spec, st, rec, waves=wO, dist=dO, seed=seed)
    assert restarts >= n and cuts >= n // 4, (restarts, cuts)


# ---- four envs per thread and the host-buffer pipeline, in a child process ------------------------------------------
N_VEC4 = 4 * 64 * 3 + 4          # 64-thread blocks of four envs per thread: the last block has one active thread
HOST_N = (4100, 4102)            # 1000-env chunks: four full chunks and a 100-env tail; 4102: every chunk one env per thread
CHILD_ENV = dict(ML4CA_ENV_VEC="4", ML4CA_ENV_THREADS="64", ML4CA_HOST_CHUNK="1000")


def step_kernel_vec(names):
    """The VEC template argument (the fourth) of every env_step_kernel name in ``names``."""
    out = set()
    for s in names:
        m = re.search(r"env_step_kernel<([^>]*)>", str(s))
        if m:
            out.add(re.sub(r"^\(\w+\)", "", m.group(1).split(",")[3].strip()))
    return out


def profiled_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages() if "env_step_kernel" in e.key})


def child(path):
    """Run with CHILD_ENV set.  Records every env class at N_VEC4 envs for the parent's oracle check, and asserts that
    step_host at HOST_N envs with per-env set-points returns exactly what a device-buffer step of a twin returns."""
    dev = torch.device("cuda", 0)
    out = {}
    for c, (kind, cont, ext) in enumerate(CLASSES):
        rng = np.random.default_rng(1000 + c)
        env = make_env(kind, cont, ext, N_VEC4, max_ep_len=L, auto_reset=True, seed=23, device=dev)
        ref, eta0, nu0, _ = setpoints_and_poses(rng, N_VEC4)
        env.set_ref(ref)
        out['%d__obs0' % c] = np_(env.reset(**init_kw(eta0, nu0)))
        box = {}
        names = profiled_kernels(lambda: box.update(run_kernel(env, rng, STEPS)))
        for k, v in box.items():
            out['%d__%s' % (c, k)] = v
        out['%d__ref' % c], out['%d__eta0' % c], out['%d__nu0' % c] = ref, eta0, nu0
        out['%d__kernels' % c] = np.array(names, dtype=str)
    for n in HOST_N:
        kw = dict(max_ep_len=L, auto_reset=True, seed=11, device=dev)
        A, B = make_env('final', True, True, n, **kw), make_env('final', True, True, n, **kw)
        ref, eta0, nu0, _ = setpoints_and_poses(np.random.default_rng(n), n)
        for e in (A, B):
            e.set_ref(ref)
            e.reset(**init_kw(eta0, nu0))
        g = torch.Generator()
        g.manual_seed(n)
        h_obs, h_rew = torch.empty(9, n).pin_memory(), torch.empty(n).pin_memory()
        h_done = torch.empty(n, dtype=torch.uint8).pin_memory()
        restarts = 0

        def steps():
            nonlocal restarts
            for t in range(STEPS):
                h_act = (torch.rand(7, n, generator=g) * 2.4 - 1.2).pin_memory()
                A.step_host(h_act, h_obs, h_rew, h_done)
                o, r, _, info = B.step(h_act.to(dev))
                torch.cuda.synchronize()
                assert torch.equal(h_obs, o.cpu()) and torch.equal(h_rew, r.cpu()), (n, t)
                assert torch.equal(h_done, info['flags'].cpu()), (n, t)
                restarts += int((h_done != 0).sum())
        out['host%d__kernels' % n] = np.array(profiled_kernels(steps), dtype=str)
        sA, sB = A.get_state(), B.get_state()
        for k in sA:
            assert torch.equal(sA[k], sB[k]), (n, k)
        assert restarts >= n, (n, restarts)
    np.savez(path, **out)


def test_vec4_and_host_pipeline_with_setpoints(cuda_device, tmp_path):
    """The four-env kernel of every env class, and the host-buffer pipeline whose chunks read the set-point rows at their
    own offset (ML4CA_ENV_VEC=4, ML4CA_ENV_THREADS=64, ML4CA_HOST_CHUNK=1000 in a child process)."""
    path = str(tmp_path / "setpoints_vec4.npz")
    subprocess.run([sys.executable, os.path.abspath(__file__), path], check=True, timeout=900, cwd=ROOT,
                   env=dict(os.environ, **CHILD_ENV))
    g = np.load(path)
    # 4100: the four-env kernel runs the chunks of the first staging slot and the tail (the second slot starts 8 bytes off
    # a 16-byte boundary at 1000-env chunks, so its chunks take the one-env kernel); 4102: every chunk one env per thread
    assert '4' in step_kernel_vec(g['host%d__kernels' % HOST_N[0]]), g['host%d__kernels' % HOST_N[0]]
    assert step_kernel_vec(g['host%d__kernels' % HOST_N[1]]) == {'1'}, g['host%d__kernels' % HOST_N[1]]
    for c, (kind, cont, ext) in enumerate(CLASSES):
        assert step_kernel_vec(g['%d__kernels' % c]) == {'4'}, (CLASS_IDS[c], g['%d__kernels' % c])
        spec = EO.EnvSpec(kind, cont, ext, max_ep_len=L)
        st = EO.new_state(spec, N_VEC4)
        st['ref'] = g['%d__ref' % c].copy()
        o_ref = EO.reset(spec, st, eta=g['%d__eta0' % c], nu=g['%d__nu0' % c])
        np.testing.assert_allclose(g['%d__obs0' % c], o_ref, rtol=0, atol=2e-5)
        rec = {k.split('__', 1)[1]: g[k] for k in g.files if k.startswith('%d__' % c)}
        restarts, cuts = check_against_oracle(spec, st, rec)
        assert restarts >= N_VEC4 and cuts >= N_VEC4 // 4, (CLASS_IDS[c], restarts, cuts)


# ---- the Python surface -----------------------------------------------------------------------------------------------
def frozen_final(n, **kw):
    import ml4ca_b200.env as E
    return E.RevoltFinal(E.StandInHull(frozen=True), extended_state=True, cont_ang=True, num_envs=n, **kw)


def oracle_obs(spec, eta, nu, ref):
    return EO.observe(spec, eta, nu, np.broadcast_to(np.asarray(ref, dtype=np.float64).reshape(3, -1), eta.shape),
                      np.zeros((3, eta.shape[1])))


def test_set_ref_broadcasts_a_vector_and_sets_rows(cuda_device):
    """set_ref([3]) sets every env to one set-point, set_ref([3, n]) each env to its own; observe() and the reset's
    observation follow, env.EF.get_pose() agrees with obs[0:3].  Kernel against kernel (observe, error frame, reset):
    4e-6, the observation tolerance of tests/test_env_gpu.py, a few ulp of the <= 16 m pose rows."""
    n = 333
    spec = EO.EnvSpec('final', True, True, n_substeps=0)
    env = frozen_final(n, device=cuda_device)
    ref, eta, nu, _ = setpoints_and_poses(np.random.default_rng(0), n)
    one = np.array([1.5, -2.25, 0.4])
    env.set_ref(one)
    assert env._ref.shape == (3, n) and (np_(env._ref) == one.astype(np.float32)[:, None]).all()
    o = env.reset(**init_kw(eta, nu))
    np.testing.assert_allclose(np_(o), oracle_obs(spec, eta, nu, one), rtol=0, atol=2e-5)
    np.testing.assert_allclose(np_(env.observe()), np_(o), rtol=0, atol=4e-6)
    np.testing.assert_allclose(np_(env.EF.get_pose()), np_(o)[0:3], rtol=0, atol=4e-6)
    env.set_ref(torch.as_tensor(ref, dtype=torch.float32, device=cuda_device))
    assert torch.equal(env.EF.get_NED_ref(), torch.as_tensor(ref, dtype=torch.float32, device=cuda_device))
    want = oracle_obs(spec, eta, nu, ref)
    np.testing.assert_allclose(np_(env.observe()), want, rtol=0, atol=2e-5)     # the state is that of the reset
    np.testing.assert_allclose(np_(env.EF.get_pose()), want[0:3], rtol=0, atol=2e-5)
    o = env.reset(**init_kw(eta, nu))
    np.testing.assert_allclose(np_(o), want, rtol=0, atol=2e-5)
    np.testing.assert_allclose(np_(env.observe()), np_(o), rtol=0, atol=4e-6)
    np.testing.assert_allclose(np_(env.EF.get_pose()), np_(o)[0:3], rtol=0, atol=4e-6)
    env.EF.update(ref=one)                                    # the reference's EF.update(ref=...) path
    np.testing.assert_allclose(np_(env.observe()), oracle_obs(spec, eta, nu, one), rtol=0, atol=2e-5)


def test_step_new_ref_takes_effect_after_the_step(cuda_device):
    """step(a, new_ref=r2) returns the observation relative to the old set-point (the wrapper updates the error frame
    after the step, customEnv.py:131); the next step is relative to r2."""
    n = 258
    spec = EO.EnvSpec('final', True, True)
    env = make_env('final', True, True, n, device=cuda_device)
    rng = np.random.default_rng(1)
    r1, eta, nu, _ = setpoints_and_poses(rng, n)
    r2, _, _, _ = setpoints_and_poses(rng, n)
    env.set_ref(r1)
    st = EO.new_state(spec, n)
    st['ref'] = r1.copy()
    EO.reset(spec, st, eta=eta, nu=nu)
    env.reset(**init_kw(eta, nu))
    for t, new_ref in enumerate((r2, None)):
        a = rng.uniform(-1, 1, (7, n)).astype(np.float32)
        o64, r64, _, _ = EO.step(spec, st, a.astype(np.float64))
        o, r, _, _ = env.step(torch.as_tensor(a, device=cuda_device), new_ref=new_ref)
        np.testing.assert_allclose(np_(o), o64, rtol=0, atol=2e-5, err_msg=str(t))
        np.testing.assert_allclose(np_(r), r64, rtol=0, atol=1e-4, err_msg=str(t))
        sg = env.get_state()
        st['eta'], st['nu'] = np_(sg['eta']).astype(np.float64), np_(sg['nu']).astype(np.float64)
        if new_ref is not None:
            st['ref'] = new_ref.copy()
    assert np.abs(r2 - r1).max() > 1.0


@pytest.mark.parametrize("testing", [True, False])
def test_reset_new_ref_only_in_testing_mode(cuda_device, testing):
    """reset(new_ref=r) applies r before the reset in testing mode and ignores it otherwise (customEnv.py:155-156)."""
    n = 64
    spec = EO.EnvSpec('final', True, True, n_substeps=0)
    env = frozen_final(n, testing=testing, device=cuda_device)
    rng = np.random.default_rng(2)
    r1, eta, nu, _ = setpoints_and_poses(rng, n)
    r2, _, _, _ = setpoints_and_poses(rng, n)
    env.set_ref(r1)
    o = env.reset(new_ref=r2, **init_kw(eta, nu))
    want = r2 if testing else r1
    np.testing.assert_array_equal(np_(env._ref), want.astype(np.float32))
    np.testing.assert_allclose(np_(o), oracle_obs(spec, eta, nu, want), rtol=0, atol=2e-5)


def test_sampled_reset_is_relative_to_the_setpoint(cuda_device):
    """A Philox reset() and a masked reset(): the sampled pose and the observation relative to each env's set-point."""
    n, seed = 1031, 5
    spec = EO.EnvSpec('final', True, True)
    env = make_env('final', True, True, n, seed=seed, device=cuda_device)
    ref, _, _, _ = setpoints_and_poses(np.random.default_rng(3), n)
    env.set_ref(ref)
    st = EO.new_state(spec, n)
    st['ref'] = ref.copy()
    want = EO.reset(spec, st, seed=seed, fraction=0.8)
    o = env.reset(fraction=0.8)
    np.testing.assert_array_equal(np_(env.get_state()['eta']), st['eta'].astype(np.float32))
    np.testing.assert_allclose(np_(o), want, rtol=0, atol=2e-5)
    np.testing.assert_allclose(np_(env.observe()), np_(o), rtol=0, atol=4e-6)
    mask = np.arange(n) % 3 == 0
    want = EO.reset(spec, st, mask=mask, seed=seed, fraction=0.5)
    o2 = env.reset(fraction=0.5, mask=mask)
    np.testing.assert_allclose(np_(o2)[:, mask], want[:, mask], rtol=0, atol=2e-5)
    np.testing.assert_array_equal(np_(o2)[:, ~mask], np_(o)[:, ~mask])


if __name__ == "__main__":
    child(sys.argv[1])
