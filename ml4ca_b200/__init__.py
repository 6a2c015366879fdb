"""ml4ca_b200 -- B200-native (sm_100a) implementation of simensov/ml4ca's dynamic-positioning hot path.

Host-side mirrors of the reference interfaces, all backed by hand-written CUDA kernels behind the
C ABI of libml4ca_b200.so (include/ml4ca_b200.h):

  env.Revolt / RevoltSimple / RevoltLimited / RevoltFinal, ErrorFrame   (specific/customEnv.py, errorFrame.py)
  qp_allocator.QPTA (solve_QP, tau_controller_callback_func)            (src/qp/ROS/qp_allocator/src/qp_allocator.py)
  core.ActorCritic / mlp_actor_critic (tcgen05 MLP forward)              (spinup/algos/tf1/ppo/core.py)
  ppo.ppo / PPOUpdater / TrajectoryBuffer, trpo.trpo / TRPOUpdater       (spinup/algos/tf1/ppo/ppo.py, trpo/trpo.py)
  pinv.pinv_pid, pinv.pinv_allocate                                      (dp_controller, absent from the reference)
  observer.DPObserver                                                    (dp_controller's state observer, absent too)
  refmodel.ReferenceModel                                                (dp_controller's reference model, absent too)

The package never imports ``oracle`` and has no CPU fallback.
"""
from . import _lib  # noqa: F401
from .env import ErrorFrame, Revolt, RevoltFinal, RevoltLimited, RevoltSimple  # noqa: F401
from .pinv import pinv_allocate, pinv_pid  # noqa: F401
from .observer import DPObserver  # noqa: F401
from .refmodel import ReferenceModel  # noqa: F401
from .qp_allocator import QPTA  # noqa: F401
from .rl_allocator import RLTA  # noqa: F401
from .core import ActorCritic, mlp_actor_critic  # noqa: F401
from .ppo import PPOUpdater, TrajectoryBuffer, ppo, rollout  # noqa: F401
from .trpo import GAEBuffer, TRPOUpdater, trpo  # noqa: F401
from .env import StandInHull  # noqa: F401
from . import evaluate  # noqa: F401

__version__ = "0.1.0"
