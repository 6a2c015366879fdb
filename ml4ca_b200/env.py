"""Batched drop-ins for the reference gym wrapper: Revolt, RevoltSimple, RevoltLimited, RevoltFinal, ErrorFrame.

Mirrors /root/reference/src/rl/windows_workspace/specific/customEnv.py (classes :11,:327,:351,:373) and
specific/errorFrame.py -- same constructor arguments, attribute names, ``reset``/``step`` signatures
and error behaviour -- but one object holds ``num_envs`` independent vessels whose state lives in HBM
and whose ``step`` is a single sm_100a kernel launch through the C ABI (ml4ca_env_step).

Batch layout is struct-of-arrays: actions ``[act_dim, num_envs]``, observations
``[obs_dim, num_envs]`` (float32, CUDA).  With ``num_envs == 1`` a flat ``(act_dim,)`` action is
accepted and flat ``(obs_dim,)`` / scalar results are returned, i.e. the reference call shape.
NumPy in -> NumPy out, torch in -> torch out.

The proprietary Cybersea simulator behind ``digitwin`` is absent from the reference; pass a
``StandInHull`` (the declared 3-DOF stand-in integrated inside the kernel) where the reference
passes a ``DigiTwin``.
"""
import ctypes

import numpy as np
import torch

from . import _lib

_KIND = {"full": 0, "revoltsimple": 1, "revoltlimited": 2, "revoltfinal": 3}


class StandInHull(object):
    """Stands where the reference passes a ``DigiTwin`` (digitwin.py:18): selects the in-kernel hull.

    frozen=True is a null simulator (the hull state only changes through reset), which isolates the
    wrapper arithmetic exactly like stepping the reference with a no-op twin.

    hull_model picks the DECLARED parameter set of the stand-in equations (ml4ca_constants.h): 0 = the default constants,
    1 = the constants fitted to the reference's recorded Cybersea box tests (tools/sysid_hull.py), which come with a
    first-order lag of the thruster wrench (actuator_lag_s, default 0.92 s for model 1 and none for model 0).
    """

    FITTED_LAG_S = 0.92         # ML4CA_H1_LAG_S

    def __init__(self, frozen=False, n_substeps=None, hull_model=0, actuator_lag_s=None):
        self.frozen = bool(frozen)
        self.n_substeps = n_substeps
        self.hull_model = int(hull_model)
        if actuator_lag_s is None:
            actuator_lag_s = self.FITTED_LAG_S if self.hull_model == 1 else 0.0
        self.actuator_lag_s = float(actuator_lag_s)


class Box(object):
    """The two attributes of gym.spaces.Box the reference's callers read (ppo.py:202-203)."""

    def __init__(self, low, high, dtype=np.float64):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.dtype = dtype
        self.shape = self.low.shape


class ErrorFrame(object):
    """errorFrame.py:4-38 for a batch: NED pose/ref ``[3, n]`` -> body-frame error ``[3, n]``.

    Keeps the training-env quirk of the reference: ``wrap_angle`` is called with its default
    ``deg=True`` on radians (mathematics.py:14, errorFrame.py:29,31), i.e. no wrap for |angle| < 180.
    """

    def __init__(self, pos=(0, 0, 0), ref=(0, 0, 0), device=None):
        self.device = torch.device(device if device is not None else "cuda")
        self._pos = self._as(pos)
        self._ref = self._as(ref)
        self._error_coordinate = None
        self.transform()

    def _as(self, x):
        t = torch.as_tensor(np.asarray(x, dtype=np.float32) if not torch.is_tensor(x) else x,
                            dtype=torch.float32, device=self.device)
        return t.reshape(3, -1).contiguous()

    def update(self, pos=None, ref=None):
        if pos is not None:
            self._pos = self._as(pos)
        if ref is not None:
            self._ref = self._as(ref)
        self.transform()

    def transform(self, pos=None):
        if pos is not None:
            self._pos = self._as(pos)
        n = max(self._pos.shape[1], self._ref.shape[1])
        pos_b = self._pos.expand(3, n).contiguous()
        ref_b = self._ref.expand(3, n).contiguous()
        err = torch.empty_like(pos_b)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_error_frame(n, _lib.ptr(pos_b), _lib.ptr(ref_b), _lib.ptr(err),
                                                    _lib.current_stream()), "ml4ca_error_frame")
        self._error_coordinate = err

    def get_pose(self, new_pose=None):
        if new_pose is not None:
            self.update(new_pose)
        return self._error_coordinate

    def get_NED_pos(self):
        return self._pos

    def get_NED_ref(self):
        return self._ref


def measured_pose(eta, nu, wave, wave_rate):
    """The measured pose and velocity a vessel's sensors report in waves (DESIGN.md section 4): the LF pose ``eta`` [3, n]
    plus the body-frame wave motion ``wave`` [3, n] rotated by the LF heading, and ``nu`` [3, n] plus ``wave_rate``.
    Host glue in torch; the env kernels compute the same sum for the observation."""
    c, s = torch.cos(eta[2]), torch.sin(eta[2])
    eta_m = torch.stack([eta[0] + c * wave[0] - s * wave[1], eta[1] + s * wave[0] + c * wave[1], eta[2] + wave[2]])
    return eta_m, nu + wave_rate


class _EnvErrorFrame(object):
    """``env.EF`` view (customEnv.py:66): reads the pose / reference held in the device-side state."""

    def __init__(self, env):
        self._env = env

    def get_NED_pos(self):
        return self._env.get_state()["eta"]

    def get_NED_ref(self):
        return self._env._ref

    def get_pose(self):
        ef = ErrorFrame(self.get_NED_pos(), self.get_NED_ref(), device=self._env.device)
        return ef.get_pose()

    def update(self, pos=None, ref=None):
        assert pos is None, "the pose belongs to the simulator; only the reference can be updated"
        if ref is not None:
            self._env.set_ref(ref)


class Revolt(object):
    """customEnv.py:11-325.  See the module docstring for the batch conventions."""

    metadata = {'render.modes': ['human']}

    def __init__(self,
                 digitwin=None,
                 num_actions=6,
                 num_states=6,
                 real_ss_bounds=(8.0, 8.0, np.pi / 2, 1.4, 0.30, 0.52),
                 testing=False,
                 realtime=False,
                 max_ep_len=800,
                 extended_state=False,
                 reset_acts=False,
                 cont_ang=False,
                 num_envs=1, device=None, seed=0, auto_reset=False, env_id_offset=0, reset_fraction=0.8):
        assert digitwin is not None, 'No digitwin was passed to Revolt environment'
        self.dTwin = digitwin
        if not hasattr(self, 'name'):
            self.name = 'full'
        self.extended_state = extended_state
        self.num_actions = num_actions
        self.num_states = num_states if not extended_state else num_states + 3
        self.num_envs = int(num_envs)
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
        self.testing = testing
        self.cont_ang = cont_ang
        self.reset_actions = reset_acts
        self.vel_rew_coeffs = [0.5, 0.5, 1.0]
        timesteps = 20
        self.n_steps = 1 if (testing and realtime) else timesteps
        self.dt = 0.01 * self.n_steps
        self.max_ep_len = int(max_ep_len * 10.0 / self.n_steps)
        self.real_ss_bounds = list(real_ss_bounds)
        self._class_defaults()

        self.action_space = Box(-1 * np.ones((self.num_actions,)), np.ones((self.num_actions,)))
        self.observation_space = Box(-1 * np.ones((self.num_states,)), np.ones((self.num_states,)))
        self.act_2_act_map_inv = getattr(self, 'act_2_act_map_inv', self.act_2_act_map)

        cfg = _lib.EnvCfg()
        kind = _KIND[self.name]
        _lib.check(_lib.lib().ml4ca_env_cfg_default(kind, int(bool(cont_ang)), int(bool(extended_state)),
                                                    ctypes.byref(cfg)), "ml4ca_env_cfg_default")
        n_sub = self.n_steps if digitwin.n_substeps is None else int(digitwin.n_substeps)
        cfg.n_substeps = 0 if digitwin.frozen else n_sub
        cfg.hull_model = int(getattr(digitwin, "hull_model", 0))
        cfg.actuator_lag_s = float(getattr(digitwin, "actuator_lag_s", 0.0))
        cfg.max_ep_len = self.max_ep_len
        cfg.auto_reset = int(bool(auto_reset))
        cfg.reset_acts = int(bool(reset_acts))            # customEnv.py:179-188
        for i in range(6):
            cfg.ss_bounds[i] = float(np.float32(self.real_ss_bounds[i]))
        cfg.step_dt = float(np.float32(self.dt))
        cfg.reset_fraction = float(reset_fraction)
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.env_id_offset = int(env_id_offset)
        self._cfg = cfg
        act_dim, obs_dim = ctypes.c_int32(), ctypes.c_int32()
        _lib.check(_lib.lib().ml4ca_env_dims(ctypes.byref(cfg), ctypes.byref(act_dim), ctypes.byref(obs_dim)))
        assert act_dim.value == self.num_actions and obs_dim.value == self.num_states
        self._handle = ctypes.c_void_p()
        _lib.check(_lib.lib().ml4ca_env_create(ctypes.byref(cfg), self.num_envs, self.device.index,
                                               ctypes.byref(self._handle)), "ml4ca_env_create")
        n = self.num_envs
        self._ref = torch.zeros(3, n, dtype=torch.float32, device=self.device)
        self._obs = torch.empty(self.num_states, n, dtype=torch.float32, device=self.device)
        self._rew = torch.empty(n, dtype=torch.float32, device=self.device)
        self._done = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._has_reset = False          # self._obs holds nothing until the first reset()
        self._disturbance = None         # the arguments of the last set_disturbance(), None = calm water
        self._waves = None               # the arguments of the last set_waves(), None = no wave motion
        self._observer = None            # the DPObserver of set_observer(), None = the agent sees the measurement
        self._refmodel = None            # the ReferenceModel of set_reference_model(), None = the set-point is the reference
        self.EF = _EnvErrorFrame(self)

    # -- per-class tables (customEnv.py:58-65); subclasses override --------------------------------
    def _class_defaults(self):
        self.default_actions = {0: 0, 1: 0, 2: 0, 3: 0, 4: 0, 5: 0}
        self.act_2_act_map = {0: 0, 1: 1, 2: 2, 3: 3, 4: 4, 5: 5}
        self.act_2_act_map_inv = self.act_2_act_map
        self.valid_action_indices = list(range(6))[0:self.num_actions]
        self.real_action_bounds = [100] * 3 + [np.pi] * 3

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            try:
                _lib.lib().ml4ca_env_destroy(h)
            except Exception:
                pass
            self._handle = None

    # -- helpers ------------------------------------------------------------------------------------
    def _to_device(self, x, rows):
        was_numpy = not torch.is_tensor(x)
        t = torch.as_tensor(np.asarray(x, dtype=np.float32) if was_numpy else x)
        t = t.to(device=self.device, dtype=torch.float32)
        flat = t.dim() == 1 and self.num_envs == 1
        t = t.reshape(rows, self.num_envs).contiguous()
        return t, was_numpy, flat

    def _out(self, t, was_numpy, flat):
        if flat:
            t = t.reshape(-1) if t.dim() == 2 else t.reshape(())
        return t.cpu().numpy().astype(np.float64) if was_numpy else t

    def _stream(self):
        return _lib.current_stream()

    def step_into(self, action, obs, rew, done):
        """The bare C-ABI call of ``step``: float32 CUDA ``action [act_dim, n]`` in, caller-owned ``obs``,
        ``rew``, ``done`` (uint8 flag byte) out.  No allocation, no extra kernels, no synchronisation."""
        _lib.check(_lib.lib().ml4ca_env_step(self._handle, _lib.ptr(action), _lib.ptr(obs), _lib.ptr(rew),
                                             _lib.ptr(done), self._stream()), "ml4ca_env_step")

    def step_host(self, action, obs, rew, done):
        """``step`` for HOST buffers (float32 CPU tensors, ideally pinned): ``action [act_dim, n]`` in, ``obs``,
        ``rew``, ``done`` (uint8 flag byte) out, through the chunked copy/compute pipeline of
        ml4ca_env_step_host.  Asynchronous: synchronise the current stream before reading the outputs."""
        for t, dt in ((action, torch.float32), (obs, torch.float32), (rew, torch.float32), (done, torch.uint8)):
            assert t.device.type == "cpu" and t.dtype == dt and t.is_contiguous(), "host buffers: contiguous CPU tensors"
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_env_step_host(self._handle, action.data_ptr(), obs.data_ptr(), rew.data_ptr(),
                                                      done.data_ptr(), self._stream()), "ml4ca_env_step_host")

    # -- gym API -------------------------------------------------------------------------------------
    def step(self, action, new_ref=None, out=None):
        """customEnv.py:92-133 -> (state, reward, done, info).

        ``done`` is the reference's ``is_terminal``; info['flags'] carries the raw flag byte
        (bit 0 terminal, bit 1 episode-length cut of ppo.py:304).  ``out=(obs, rew, done)`` lets the
        caller supply the output tensors (no allocation on the step path).
        """
        a, was_numpy, flat = self._to_device(action, self.num_actions)
        obs, rew, done = out if out is not None else (torch.empty_like(self._obs), torch.empty_like(self._rew),
                                                      torch.empty_like(self._done))
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_env_step(self._handle, _lib.ptr(a), _lib.ptr(obs), _lib.ptr(rew),
                                                 _lib.ptr(done), self._stream()), "ml4ca_env_step")
        if new_ref is not None:
            self.EF.update(ref=new_ref)   # :131
        self._obs = obs                   # the observation of "the last reset() / step()" (rollout(), masked reset())
        info = {'None': 0, 'flags': done}
        d = (done & 1).bool()
        if flat:
            return self._out(obs, was_numpy, True), self._out(rew, was_numpy, True), bool(d.item()), info
        if was_numpy:
            return self._out(obs, True, False), self._out(rew, True, False), d.cpu().numpy(), info
        return obs, rew, d, info

    def reset(self, new_ref=None, fraction=0.8, fixed_point=None, mask=None, as_numpy=False, **init):
        """customEnv.py:135-194 -> initial observation.

        ``init`` takes the reference keys 'Hull.PosNED' [N, E], 'Hull.PosAttitude' [0, 0, yaw],
        'Hull.VelocityNu' [u, v, 0, 0, 0, r]; entries may be scalars or per-env arrays.
        ``mask`` (bool [num_envs]) restricts the reset to a subset (the caller-side reset of
        finished envs in a batched rollout).
        """
        n = self.num_envs
        m = None
        if mask is not None:
            m = torch.as_tensor(mask).to(device=self.device).to(torch.uint8).contiguous()
        obs = self._obs
        if self.testing and new_ref is not None:      # :155-156
            self.EF.update(ref=new_ref)
        eta = nu = None
        if init:
            ned = np.broadcast_to(np.asarray(init.get('Hull.PosNED', [0, 0]), dtype=np.float64).reshape(2, -1), (2, n))
            att = np.asarray(init.get('Hull.PosAttitude', [0, 0, 0]), dtype=np.float64).reshape(3, -1)
            vel = np.asarray(init.get('Hull.VelocityNu', [0] * 6), dtype=np.float64).reshape(6, -1)
            eta = np.stack([ned[0], ned[1], np.broadcast_to(att[2], (n,))])
            nu = np.stack([np.broadcast_to(vel[0], (n,)), np.broadcast_to(vel[1], (n,)), np.broadcast_to(vel[5], (n,))])
        elif self.testing:                            # :146-150, simtools.py:81-107
            eta = np.zeros((3, n))
            if fixed_point is None:
                theta = np.random.random(n) * 2 * np.pi
                eta[1], eta[0] = 5 * np.cos(theta), 5 * np.sin(theta)
                eta[2] = np.random.uniform(-5 * np.pi / 180, 5 * np.pi / 180, n)
            else:
                thetas = [0.0, np.pi / 4, np.pi / 2, np.pi, 5 * np.pi / 4, 3 * np.pi / 2]
                angles = [0.0, 0.0, -15.0, 15.0, 0.0, -15.0]
                k = fixed_point % len(thetas)
                ang = np.pi / 2 - thetas[k]
                eta[1], eta[0], eta[2] = 5 * np.cos(ang), 5 * np.sin(ang), angles[k] * np.pi / 180
            nu = np.zeros((3, n))
        with torch.cuda.device(self.device):
            if eta is not None:
                eta_t = torch.as_tensor(eta, dtype=torch.float32, device=self.device).contiguous()
                nu_t = torch.as_tensor(nu, dtype=torch.float32, device=self.device).contiguous()
                _lib.check(_lib.lib().ml4ca_env_reset_to(self._handle, _lib.ptr(m), _lib.ptr(eta_t), _lib.ptr(nu_t),
                                                         _lib.ptr(obs), self._stream()), "ml4ca_env_reset_to")
            else:
                _lib.check(_lib.lib().ml4ca_env_reset(self._handle, _lib.ptr(m), float(fraction), _lib.ptr(obs),
                                                      self._stream()), "ml4ca_env_reset")
        if m is None:
            self._has_reset = True
        out = obs.clone()                 # columns outside `mask` keep the observation of the last step()
        if self.num_envs == 1 and (as_numpy or bool(init)):
            return out.reshape(-1).cpu().numpy().astype(np.float64)
        return out.cpu().numpy().astype(np.float64) if as_numpy else out

    def render(self):
        pass

    # -- state access ----------------------------------------------------------------------------------
    def set_ref(self, ref):
        r = torch.as_tensor(np.asarray(ref, dtype=np.float32) if not torch.is_tensor(ref) else ref,
                            dtype=torch.float32, device=self.device).reshape(3, -1)
        self._ref = r.expand(3, self.num_envs).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_env_set_ref(self._handle, _lib.ptr(self._ref), self._stream()))

    def set_reset_fraction(self, fraction):
        """The ``fraction`` in-kernel restarts sample with (auto_reset; the reference passes it per reset, ppo.py:319-322)."""
        self._cfg.reset_fraction = float(fraction)
        _lib.check(_lib.lib().ml4ca_env_set_reset_fraction(self._handle, float(fraction)), "ml4ca_env_set_reset_fraction")

    def set_disturbance(self, current_speed=(0.0, 0.0), current_direction=(0.0, 2 * np.pi), bias_std=(0.0, 0.0, 0.0),
                        bias_time_s=0.0):
        """Environmental loads (the declared model of DESIGN.md section 4); ``set_disturbance(None)`` is calm water again.

        Every reset (explicit or in-kernel) draws an ocean current, constant in the NED frame over the episode, with speed
        ~ U(current_speed) m/s and direction ~ U(current_direction) rad (the direction the water flows towards: 0 = north,
        pi/2 = east), and a NED bias force b = [X_N, Y_E, N_psi] (N, N, Nm) with standard deviation ``bias_std``.  b follows
        a first-order Gauss-Markov process with time constant ``bias_time_s`` (0 = constant over the episode).  Enabling
        draws the state of every env at once.  0 to 0.2 m/s is the useful current range: a 0.3 m/s beam current takes all
        of the sway thrust.  Like the restart fraction, the setting is a launch parameter: CUDA graphs captured earlier
        keep theirs."""
        with torch.cuda.device(self.device):
            if current_speed is None:
                _lib.check(_lib.lib().ml4ca_env_set_disturbance(self._handle, None, self._stream()), "ml4ca_env_set_disturbance")
                self._disturbance = None
                return
            c = _lib.DisturbanceCfg()
            c.current_speed_min, c.current_speed_max = (float(x) for x in current_speed)
            c.current_dir_min, c.current_dir_max = (float(x) for x in current_direction)
            for i, x in enumerate(bias_std):
                c.bias_std[i] = float(x)
            c.bias_time_s = float(bias_time_s)
            _lib.check(_lib.lib().ml4ca_env_set_disturbance(self._handle, ctypes.byref(c), self._stream()),
                       "ml4ca_env_set_disturbance")
        self._disturbance = (tuple(current_speed), tuple(current_direction), tuple(bias_std), float(bias_time_s))

    def set_disturbance_state(self, current=None, bias=None):
        """Overwrite the disturbance state: ``current`` [2, num_envs] (NED, m/s), ``bias`` [3, num_envs] (N, N, Nm); either
        may be None.  The values hold until that env's next reset."""
        cur = None if current is None else self._to_device(current, 2)[0]
        b = None if bias is None else self._to_device(bias, 3)[0]
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_env_set_disturbance_state(self._handle, _lib.ptr(cur), _lib.ptr(b), self._stream()),
                       "ml4ca_env_set_disturbance_state")

    def set_waves(self, sigma=(0.0, 0.0, 0.0), peak_frequency=(1.0, 2.0), damping=0.1):
        """First-order wave-frequency motion (the declared model of DESIGN.md section 4); ``set_waves(None)`` switches it off.

        Per env and DOF (surge, sway, yaw; body frame) a second-order oscillator driven by white noise with stationary
        std ``sigma`` (m, m, rad), damping ratio ``damping`` and peak frequency w0 ~ U(peak_frequency) rad/s, drawn at every
        reset (explicit or in-kernel) together with a stationary state.  The motion never moves the hull: ``get_state()``'s
        "eta" and "nu" stay the low-frequency state, while the observation, reward and termination of every step and reset
        (and ``observe()``) see the measured pose and velocity, LF plus wave motion.  Enabling draws the state of every env
        at once.  Like the disturbance, the setting is a launch parameter: CUDA graphs captured earlier keep theirs."""
        with torch.cuda.device(self.device):
            if sigma is None:
                _lib.check(_lib.lib().ml4ca_env_set_waves(self._handle, None, self._stream()), "ml4ca_env_set_waves")
                self._waves = None
                return
            c = _lib.WaveCfg()
            for i, x in enumerate(sigma):
                c.sigma[i] = float(x)
            c.omega_min, c.omega_max = (float(x) for x in peak_frequency)
            c.damping = float(damping)
            _lib.check(_lib.lib().ml4ca_env_set_waves(self._handle, ctypes.byref(c), self._stream()), "ml4ca_env_set_waves")
        self._waves = (tuple(float(x) for x in sigma), tuple(float(x) for x in peak_frequency), float(damping))

    def set_wave_state(self, motion=None, rate=None, omega=None):
        """Overwrite the wave state: ``motion`` [3, num_envs] (m, m, rad), ``rate`` [3, num_envs] (m/s, m/s, rad/s), both in
        the body frame, and ``omega`` [num_envs] (rad/s); any may be None.  The values hold until that env's next reset."""
        x = None if motion is None else self._to_device(motion, 3)[0]
        xd = None if rate is None else self._to_device(rate, 3)[0]
        w = None if omega is None else self._to_device(omega, 1)[0]
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_env_set_wave_state(self._handle, _lib.ptr(x), _lib.ptr(xd), _lib.ptr(w), self._stream()),
                       "ml4ca_env_set_wave_state")

    def set_observer(self, observer):
        """Run a ``DPObserver`` in the loop (DESIGN.md section 4, "DP observer in the loop"); ``set_observer(None)`` detaches.

        While attached, every step advances the observer inside the step kernel, on the measured pose after the step and
        the thrust and azimuths the step applied, and the observation rows 0-5 become the body-frame error of the estimated
        pose eta^ and the estimated velocity nu^: what the controller of a DP vessel sees.  Rows 6-8, the reward, the
        termination and the vessel itself are unchanged.  Every reset and in-kernel restart re-initialises the observer
        of that env on its new measured pose.  Attaching re-initialises every env's observer on its current measured pose.
        ``observer`` must have this env's num_envs, device and step; its hull model may differ.  The env keeps a reference:
        the observer's ``state`` and ``omega_o`` tensors are read and written by every step.  Like the waves, the setting
        is a launch parameter: ``rollout()`` keys its captured graphs on it."""
        with torch.cuda.device(self.device):
            if observer is None:
                _lib.check(_lib.lib().ml4ca_env_set_observer(self._handle, None, None, None, self._stream()),
                           "ml4ca_env_set_observer")
            else:
                assert observer.num_envs == self.num_envs, "the observer has %d envs, the env %d" % (observer.num_envs,
                                                                                                   self.num_envs)
                assert observer.state.device == self.device and observer.omega_o.device == self.device, \
                    "the observer lives on %s, the env on %s" % (observer.state.device, self.device)
                _lib.check(_lib.lib().ml4ca_env_set_observer(self._handle, ctypes.byref(observer.cfg), _lib.ptr(observer.state),
                                                             _lib.ptr(observer.omega_o), self._stream()),
                           "ml4ca_env_set_observer")
        self._observer = observer
        if self._has_reset:             # rows 0-5 of the last observation now come from the estimates (or the measurement)
            if observer is not None:
                eta, nu = observer.eta_hat.contiguous(), observer.nu_hat.contiguous()
            else:
                st = self.get_state()
                eta, nu = (st["eta_measured"], st["nu_measured"]) if "eta_measured" in st else (st["eta"], st["nu"])
            obs = self._obs.clone()
            obs[0:3] = ErrorFrame(eta, self._obs_ref(), device=self.device).get_pose()
            obs[3:6] = nu
            self._obs = obs

    def _obs_ref(self):
        """What observation rows 0-2 are formed against: eta_d of an attached reference model, else the set-point."""
        return self._ref if self._refmodel is None else self._refmodel.eta_d.contiguous()

    def set_reference_model(self, model):
        """Run a ``ReferenceModel`` in the loop (DESIGN.md section 4, "DP reference model in the loop");
        ``set_reference_model(None)`` detaches.

        While attached, the set-point (``set_ref``, ``step(new_ref=)``) is the operator's command s, and every step first
        advances the model once on s inside the step kernel; the observation rows 0-2, the reward and the termination are
        then formed against the model's eta_d instead of s, so the agent is trained and evaluated on tracking a smooth
        reference.  Rows 3-8 are unchanged (the reward's velocity penalty still acts on nu, not nu - v_d).  Every reset and
        in-kernel restart starts that env's model again at its new LF pose (eta_d = eta, v_d = a_d = 0); attaching starts
        every env's model at its current LF pose.  ``model`` must have this env's num_envs, device and step.  The env keeps
        a reference: the model's ``state`` is read and written by every step, so ``eta_d`` / ``v_d`` / ``a_d`` show the
        in-loop values.  Like the observer, the setting is a launch parameter: ``rollout()`` keys its captured graphs on
        it."""
        with torch.cuda.device(self.device):
            if model is None:
                _lib.check(_lib.lib().ml4ca_env_set_refmodel(self._handle, None, None, self._stream()),
                           "ml4ca_env_set_refmodel")
            else:
                assert model.num_envs == self.num_envs, "the reference model has %d envs, the env %d" % (model.num_envs,
                                                                                                         self.num_envs)
                assert model.state.device == self.device, \
                    "the reference model lives on %s, the env on %s" % (model.state.device, self.device)
                _lib.check(_lib.lib().ml4ca_env_set_refmodel(self._handle, ctypes.byref(model.cfg), _lib.ptr(model.state),
                                                             self._stream()), "ml4ca_env_set_refmodel")
        self._refmodel = model
        if self._has_reset:             # rows 0-2 of the last observation are now formed against eta_d (or the set-point)
            if self._observer is not None:
                eta = self._observer.eta_hat.contiguous()
            else:
                st = self.get_state()
                eta = st.get("eta_measured", st["eta"])
            obs = self._obs.clone()
            obs[0:3] = ErrorFrame(eta, self._obs_ref(), device=self.device).get_pose()
            self._obs = obs

    def observe(self):
        """state() / state_extended() (customEnv.py:196-205) of the current device-side state (measured, with waves on;
        rows 0-5 from the estimates while an observer is attached; rows 0-2 against eta_d while a reference model is
        attached)."""
        obs = torch.empty_like(self._obs)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_env_observe(self._handle, _lib.ptr(obs), self._stream()), "ml4ca_env_observe")
        return obs

    def get_state(self):
        n = self.num_envs
        f = lambda rows: torch.empty(rows, n, dtype=torch.float32, device=self.device)
        st = {"eta": f(3), "nu": f(3), "prev_thrust": f(3), "angles": f(3),
              "ep_len": torch.empty(n, dtype=torch.int32, device=self.device)}
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_env_get_state(self._handle, _lib.ptr(st["eta"]), _lib.ptr(st["nu"]),
                                                      _lib.ptr(st["prev_thrust"]), _lib.ptr(st["angles"]),
                                                      _lib.ptr(st["ep_len"]), self._stream()))
            if self._disturbance is not None:   # current [2, n] (NED, m/s) and bias [3, n] (N, N, Nm) of the episode
                st["current"], st["bias"] = f(2), f(3)
                _lib.check(_lib.lib().ml4ca_env_get_disturbance(self._handle, _lib.ptr(st["current"]), _lib.ptr(st["bias"]),
                                                                self._stream()), "ml4ca_env_get_disturbance")
            if self._waves is not None:         # wave motion [3, n], rate [3, n] (body frame), peak frequency [n]
                st["wave"], st["wave_rate"] = f(3), f(3)
                st["wave_omega"] = torch.empty(n, dtype=torch.float32, device=self.device)
                _lib.check(_lib.lib().ml4ca_env_get_waves(self._handle, _lib.ptr(st["wave"]), _lib.ptr(st["wave_rate"]),
                                                          _lib.ptr(st["wave_omega"]), self._stream()), "ml4ca_env_get_waves")
                st["eta_measured"], st["nu_measured"] = measured_pose(st["eta"], st["nu"], st["wave"], st["wave_rate"])
        return st

    @property
    def prev_thrust(self):
        return self.get_state()["prev_thrust"]

    @property
    def current_angles(self):
        return self.get_state()["angles"]

    # -- action post-processing, also used by evaluation code (test_policy.py:135-145) ----------------
    def scale_and_clip(self, action, return_saturation=False):
        """customEnv.py:215-225 (after the angle transform of :104-108 for the final env)."""
        a, was_numpy, flat = self._to_device(action, self.num_actions)
        k = len(self.real_action_bounds)
        out = torch.empty(k, self.num_envs, dtype=torch.float32, device=self.device)
        sat = torch.empty(k, self.num_envs, dtype=torch.int8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_scale_and_clip(ctypes.byref(self._cfg), self.num_envs, _lib.ptr(a),
                                                       _lib.ptr(out), _lib.ptr(sat), self._stream()))
        res = self._out(out, was_numpy, flat)
        if flat and was_numpy:
            res = res.tolist()
        return (res, sat) if return_saturation else res

    def handle_continuous_angles(self, action):
        """customEnv.py:227-235: [a0, a1, a2, atan2(a3, a4)/pi, atan2(a5, a6)/pi] (host-side helper)."""
        assert self.name.lower() == 'revoltfinal' and self.cont_ang is True, \
            'Using continuous angles is only made to work with the final environment fully rotating stern thrusters'
        a = np.asarray(action.cpu() if torch.is_tensor(action) else action, dtype=np.float64)
        bnd = self.real_action_bounds[3]
        return np.concatenate([a[0:3], [np.arctan2(a[3], a[4]) / bnd, np.arctan2(a[5], a[6]) / bnd]])


class RevoltSimple(Revolt):
    """customEnv.py:327-349: fixed azimuths, three thrust actions."""

    def __init__(self, digitwin, testing=False, realtime=False, max_ep_len=800, extended_state=False,
                 reset_acts=False, cont_ang=False, **batch):
        self.name = 'revoltsimple'
        assert not extended_state, \
            'RevoltSimple + extended state fails in the reference too (IndexError at customEnv.py:319)'
        super().__init__(digitwin=digitwin, num_actions=3, num_states=6,
                         real_ss_bounds=[8.0, 8.0, np.pi / 2, 1.75, 0.30, 0.51], testing=testing, realtime=realtime,
                         max_ep_len=max_ep_len, extended_state=extended_state, reset_acts=reset_acts, cont_ang=False,
                         **batch)

    def _class_defaults(self):
        self.real_action_bounds = [100] * 3
        self.default_actions = {0: 0, 1: 0, 2: 0, 3: np.pi / 2, 4: -3 * np.pi / 4, 5: 3 * np.pi / 4}
        self.act_2_act_map = {0: 0, 1: 1, 2: 2}
        self.act_2_act_map_inv = self.act_2_act_map
        self.valid_action_indices = [0, 1, 2]


class RevoltLimited(Revolt):
    """customEnv.py:351-371: stern azimuths limited to +-90 deg, bow fixed."""

    def __init__(self, digitwin, testing=False, realtime=False, max_ep_len=800, extended_state=False,
                 reset_acts=False, cont_ang=False, **batch):
        self.name = 'revoltlimited'
        assert not cont_ang, 'continuous angles only work with the final environment (customEnv.py:228)'
        super().__init__(digitwin=digitwin, num_actions=5, num_states=6,
                         real_ss_bounds=[8.0, 8.0, 45 * np.pi / 180, 1.4, 0.30, 0.52], testing=testing,
                         realtime=realtime, max_ep_len=max_ep_len, extended_state=extended_state,
                         reset_acts=reset_acts, cont_ang=False, **batch)

    def _class_defaults(self):
        self.real_action_bounds = [100] * 3 + [np.pi / 2] * 2
        self.valid_action_indices = [0, 1, 2, 4, 5]
        self.act_2_act_map = {0: 0, 1: 1, 2: 2, 4: 3, 5: 4}
        self.act_2_act_map_inv = {0: 0, 1: 1, 2: 2, 3: 4, 4: 5}
        self.default_actions = {0: 0, 1: 0, 2: 0, 3: np.pi / 2, 4: 0, 5: 0}


class RevoltFinal(Revolt):
    """customEnv.py:373-399: fully rotating stern azimuths; 7 actions with continuous angles."""

    def __init__(self, digitwin, testing=False, realtime=False, max_ep_len=800, extended_state=False,
                 reset_acts=False, cont_ang=False, **batch):
        self.name = 'revoltfinal'
        n_actions = 7 if cont_ang else 5
        super().__init__(digitwin=digitwin, num_actions=n_actions, num_states=6,
                         real_ss_bounds=[8.0, 8.0, 45 * np.pi / 180, 1.4, 0.30, 0.52], testing=testing,
                         realtime=realtime, max_ep_len=max_ep_len, extended_state=extended_state,
                         reset_acts=reset_acts, cont_ang=cont_ang, **batch)

    def _class_defaults(self):
        self.real_action_bounds = [100] * 3 + [np.pi] * 2
        self.valid_action_indices = [0, 1, 2, 4, 5]
        self.act_2_act_map = {0: 0, 1: 1, 2: 2, 4: 3, 5: 4}
        self.act_2_act_map_inv = {0: 0, 1: 1, 2: 2, 3: 4, 4: 5}
        self.default_actions = {0: 0, 1: 0, 2: 0, 3: np.pi / 2, 4: 0, 5: 0}
