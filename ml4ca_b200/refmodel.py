"""DP reference model for a batch of vessels (ml4ca_refmodel_step; DESIGN.md section 4, "DP reference model").

A DP system puts a reference model (guidance) between the operator's set-point and the controller: it turns a step in
the set-point into a smooth desired pose eta_d, with a desired velocity v_d and acceleration a_d inside declared limits,
so the controller is never asked for more than the thrusters deliver.  Per env and per DOF (N, E, psi; NED) it is a
third-order filter with saturating elements (Fossen 2011, section 12.1).  The reference's DP stack (dp_controller)
assumes one and does not contain it, like the PID and the observer.

State layout: ``state`` [9, n] float32 with rows eta_d[0:3] (N, E, psi; psi not wrapped), v_d[3:6] (NED rates),
a_d[6:9].
"""
import ctypes

import torch

from . import _lib

_PARAMS = ("zeta", "omega", "v_max", "a_max")


class ReferenceModel(object):
    """``num_envs`` reference filters on ``device``, advanced once per env step of ``step_dt`` seconds.  ``overrides``: any
    of zeta, omega (rad/s), v_max (m/s, m/s, rad/s), a_max (m/s^2, m/s^2, rad/s^2), 3 values each (N, E, psi); the rest
    are the declared defaults of ``ml4ca_refmodel_cfg_default``.  A configuration the kernel rejects (non-positive values,
    an unstable sub-step map) raises at the first ``step``."""

    def __init__(self, num_envs, step_dt=0.2, device=None, **overrides):
        unknown = set(overrides) - set(_PARAMS)
        assert not unknown, "unknown reference model parameters: %s" % sorted(unknown)
        self.num_envs = int(num_envs)
        self.device = torch.device(device if device is not None else "cuda")
        cfg = _lib.RefModelCfg()
        _lib.check(_lib.lib().ml4ca_refmodel_cfg_default(ctypes.byref(cfg)), "ml4ca_refmodel_cfg_default")
        cfg.step_dt = float(step_dt)
        for k, v in overrides.items():
            for d, x in enumerate(v):
                getattr(cfg, k)[d] = float(x)
        self.cfg = cfg
        self.state = torch.zeros(9, self.num_envs, dtype=torch.float32, device=self.device)

    @classmethod
    def for_env(cls, env, **kw):
        """A reference model matching a ``Revolt`` env: its num_envs, step (env.dt) and device."""
        kw.setdefault("step_dt", float(env.dt))
        kw.setdefault("device", env.device)
        return cls(env.num_envs, **kw)

    @property
    def step_dt(self):
        return float(self.cfg.step_dt)

    def _rows(self, t):
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device)
        return t.reshape(3, -1).expand(3, self.num_envs).contiguous()

    def reset(self, eta0):
        """eta_d = eta0 ([3] or [3, n]), v_d = a_d = 0."""
        eta0 = self._rows(eta0)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_refmodel_reset(self.num_envs, _lib.ptr(eta0), _lib.ptr(self.state),
                                                       _lib.current_stream()), "ml4ca_refmodel_reset")

    def step(self, setpoint):
        """One env step toward ``setpoint`` ([3] or [3, n]: N, E, psi), held over the step.  Returns views (eta_d, v_d)."""
        r = self._rows(setpoint)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_refmodel_step(ctypes.byref(self.cfg), self.num_envs, _lib.ptr(r),
                                                      _lib.ptr(self.state), _lib.current_stream()), "ml4ca_refmodel_step")
        return self.eta_d, self.v_d

    @property
    def eta_d(self):
        return self.state[0:3]

    @property
    def v_d(self):
        return self.state[3:6]

    @property
    def a_d(self):
        return self.state[6:9]
