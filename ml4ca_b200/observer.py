"""Passive nonlinear DP observer for a batch of vessels (ml4ca_observer_step; DESIGN.md section 4, "DP observer").

A DP system puts a state observer between the sensors and the controller: from the measured pose (in waves: the
low-frequency pose plus the wave-frequency motion) and the thrust the vessel applied, it estimates the wave-filtered
pose, the low-frequency body velocity and the slowly varying environmental force.  The reference's DP stack
(dp_controller) assumes one and does not contain it, like the PID.

State layout: ``state`` [15, n] float32 with rows xi1^[0:3], xi2^[3:6] (the wave-frequency pose estimate), eta^[6:9]
(N, E, psi), nu^[9:12] (u, v, r), b^[12:15] (NED: N, N, Nm, the frame and units of ``Revolt.get_state()["bias"]``).
"""
import ctypes

import torch

from . import _lib

_GAINS = ("notch_damping", "wave_damping", "cutoff_ratio", "bias_time_s", "k3", "k4")


class DPObserver(object):
    """``num_envs`` observers on ``device``.  ``peak_frequency`` (rad/s) fills ``omega_o``, the observer's wave peak
    frequency per env: keep it (a vessel's fixed tuning) or overwrite it, e.g. with ``env.get_state()["wave_omega"]``.
    Values outside [0.1, 10] rad/s (NaN included) are clamped by the kernel.  ``gain_overrides``: any of
    notch_damping, wave_damping, cutoff_ratio, bias_time_s (0 = infinity) and the per-DOF k3, k4 (3 values each); the
    rest are the declared defaults of ``ml4ca_observer_cfg_default(hull_model)``."""

    def __init__(self, num_envs, step_dt=0.2, hull_model=0, peak_frequency=1.5, device=None, **gain_overrides):
        unknown = set(gain_overrides) - set(_GAINS)
        assert not unknown, "unknown observer gains: %s" % sorted(unknown)
        self.num_envs = int(num_envs)
        self.device = torch.device(device if device is not None else "cuda")
        cfg = _lib.ObserverCfg()
        _lib.check(_lib.lib().ml4ca_observer_cfg_default(int(hull_model), ctypes.byref(cfg)), "ml4ca_observer_cfg_default")
        cfg.step_dt = float(step_dt)
        for k, v in gain_overrides.items():
            if k in ("k3", "k4"):
                for d, x in enumerate(v):
                    getattr(cfg, k)[d] = float(x)
            else:
                setattr(cfg, k, float(v))
        self.cfg = cfg
        n = self.num_envs
        self.state = torch.zeros(15, n, dtype=torch.float32, device=self.device)
        self.omega_o = torch.full((n,), float(peak_frequency), dtype=torch.float32, device=self.device)

    @classmethod
    def for_env(cls, env, **kw):
        """An observer matching a ``Revolt`` env: its num_envs, step (env.dt), hull model and device."""
        kw.setdefault("step_dt", float(env.dt))
        kw.setdefault("hull_model", int(env._cfg.hull_model))
        kw.setdefault("device", env.device)
        return cls(env.num_envs, **kw)

    def _rows(self, t, rows):
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device)
        return t.reshape(rows, self.num_envs).contiguous()

    def _mask(self, m):
        return None if m is None else torch.as_tensor(m, device=self.device).to(torch.uint8).reshape(self.num_envs).contiguous()

    def reset(self, y, mask=None):
        """eta^ = y [3, n], the other states zero, for every env (or those where ``mask`` is non-zero)."""
        y, m = self._rows(y, 3), self._mask(mask)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_observer_reset(self.num_envs, _lib.ptr(y), _lib.ptr(m), _lib.ptr(self.state),
                                                       _lib.current_stream()), "ml4ca_observer_reset")

    def step(self, y, thrust, angles, restart=None):
        """One env step: y [3, n] measured after the step, thrust [3, n] (%) and angles [3, n] (rad) that step applied, env
        order bow, port, star (``get_state()["prev_thrust"]``, ``["angles"]``).  ``restart`` [n] (e.g. the done-flag byte
        under auto_reset): those envs are re-initialised from y instead.  Returns views (eta_hat, nu_hat, bias_hat)."""
        y, th, an, m = self._rows(y, 3), self._rows(thrust, 3), self._rows(angles, 3), self._mask(restart)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_observer_step(ctypes.byref(self.cfg), self.num_envs, _lib.ptr(y), _lib.ptr(th),
                                                      _lib.ptr(an), _lib.ptr(self.omega_o), _lib.ptr(m), _lib.ptr(self.state),
                                                      _lib.current_stream()), "ml4ca_observer_step")
        return self.eta_hat, self.nu_hat, self.bias_hat

    @property
    def eta_hat(self):
        return self.state[6:9]

    @property
    def nu_hat(self):
        return self.state[9:12]

    @property
    def bias_hat(self):
        return self.state[12:15]

    def get_state(self):
        """Copies of the estimates: "eta" [3, n], "nu" [3, n], "bias" [3, n] (NED) and "wave" [3, n] (xi2^, the estimated
        wave-frequency pose)."""
        return {"eta": self.state[6:9].clone(), "nu": self.state[9:12].clone(), "bias": self.state[12:15].clone(),
                "wave": self.state[3:6].clone()}
