"""Pseudoinverse thrust allocation + DP PID controller (batched, one CUDA thread per vessel).

This component is ABSENT from the reference (DNV GL's private ``dp_controller`` ROS package:
``nodesThruster_allocation.py`` / ``DP_PID.py``, referenced at
src/qp/ROS/qp_allocator/src/qp_allocator.py:6,83 and src/sl/SupervisedTau.py:37).  The equations are
this build's own, stated in DESIGN.md and in csrc/pinv_pid.cu; parity is unpinned.
"""
import torch

from . import _lib


def _f32(x, rows, device):
    t = torch.as_tensor(x, dtype=torch.float32, device=device)
    return t.reshape(rows, -1).contiguous()


def pinv_allocate(tau, device=None):
    """tau [3, n] (surge force, sway force, yaw moment) -> (n_pct [3, n] percent in allocator order
    port, star, bow; alpha [2, n] stern azimuths in rad).  Bow azimuth is fixed at pi/2."""
    device = torch.device(device if device is not None else (tau.device if torch.is_tensor(tau) else "cuda"))
    tau = _f32(tau, 3, device)
    n = tau.shape[1]
    n_pct = torch.empty(3, n, dtype=torch.float32, device=device)
    alpha = torch.empty(2, n, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        _lib.check(_lib.lib().ml4ca_pinv_allocate(n, _lib.ptr(tau), _lib.ptr(n_pct), _lib.ptr(alpha),
                                                  _lib.current_stream()), "ml4ca_pinv_allocate")
    return n_pct, alpha


def pinv_pid(eta, nu, ref, integ, device=None, return_tau=False, nu_d=None):
    """One DP control step: PID on the body-frame error, then pseudoinverse allocation.

    eta, nu, ref [3, n]; integ [3, n] float32 CUDA tensor updated IN PLACE (integral state).
    nu_d [3, n]: velocity feed-forward, the desired NED rates of a reference model (``ReferenceModel.v_d``); the D-term
    then acts on nu - R(psi)^T nu_d (ml4ca_pinv_pid_ff).
    Returns (n_pct [3, n], alpha [2, n]) and the saturated wrench tau [3, n] if return_tau.
    """
    assert torch.is_tensor(integ) and integ.is_cuda and integ.dtype == torch.float32 and integ.is_contiguous(), \
        "integ must be a contiguous float32 CUDA tensor (it is updated in place)"
    device = integ.device
    eta, nu, ref = _f32(eta, 3, device), _f32(nu, 3, device), _f32(ref, 3, device)
    n = eta.shape[1]
    assert integ.shape == (3, n)
    n_pct = torch.empty(3, n, dtype=torch.float32, device=device)
    alpha = torch.empty(2, n, dtype=torch.float32, device=device)
    tau = torch.empty(3, n, dtype=torch.float32, device=device) if return_tau else None
    with torch.cuda.device(device):
        if nu_d is None:
            _lib.check(_lib.lib().ml4ca_pinv_pid(n, _lib.ptr(eta), _lib.ptr(nu), _lib.ptr(ref), _lib.ptr(integ),
                                                 _lib.ptr(tau), _lib.ptr(n_pct), _lib.ptr(alpha),
                                                 _lib.current_stream()), "ml4ca_pinv_pid")
        else:
            nu_d = _f32(nu_d, 3, device)
            assert nu_d.shape == (3, n)
            _lib.check(_lib.lib().ml4ca_pinv_pid_ff(n, _lib.ptr(eta), _lib.ptr(nu), _lib.ptr(ref), _lib.ptr(nu_d),
                                                    _lib.ptr(integ), _lib.ptr(tau), _lib.ptr(n_pct), _lib.ptr(alpha),
                                                    _lib.current_stream()), "ml4ca_pinv_pid_ff")
    return (n_pct, alpha, tau) if return_tau else (n_pct, alpha)
