"""GPU parity of K2 (pseudoinverse allocation + DP PID) against the float64 oracle of the same declared
equations (the reference holds no implementation: parity unpinned, see oracle/pinv_oracle.py)."""
import numpy as np
import pytest
import torch

from oracle import pinv_oracle as PO
from oracle import constants as C

pytestmark = pytest.mark.gpu


def setpoint_batch(n, seed):
    """Per-env set-points N, E ~ U(+-4 m), psi ~ U(+-0.6 rad), and the pose of synth_batch with every fourth env turned
    round: its heading and its set-point heading on either side of +-pi (|psi - psi_ref| ~ 2 pi - 0.6 .. 2 pi), so that
    the PID's wrap_rad(psi - psi_ref) has to wrap.  float32 values."""
    eta, nu, _, _ = PO.synth_batch(n, seed=seed)
    rng = np.random.default_rng(seed + 100)
    ref = rng.uniform(-1, 1, (3, n)) * np.array([[4.0], [4.0], [0.6]])
    far = np.arange(n) % 4 == 1
    side = np.where(rng.random(n) < 0.5, 1.0, -1.0)
    eta[2, far] = -side[far] * (np.pi - rng.uniform(0, 0.3, far.sum()))
    ref[2, far] = side[far] * (np.pi - rng.uniform(0, 0.3, far.sum()))
    return eta.astype(np.float32), nu.astype(np.float32), ref.astype(np.float32)


@pytest.mark.parametrize("n", [1, 5, 4096, 1 << 20])
def test_pinv_pid_matches_oracle(cuda_device, n):
    """At the origin (the set-point of synth_batch) and at per-env set-points with headings either side of +-pi; n even
    runs the two-envs-per-thread kernel, n odd the scalar one."""
    import ml4ca_b200 as M
    origin = tuple(x.astype(np.float32) for x in PO.synth_batch(n, seed=1)[0:3])
    for eta, nu, ref in (origin, setpoint_batch(n, 2)):
        check_pinv_pid(M, cuda_device, n, eta, nu, ref)


def check_pinv_pid(M, cuda_device, n, eta, nu, ref):
    integ_t = torch.zeros(3, n, device=cuda_device)
    want_integ = np.zeros((3, n))
    for it in range(2):
        n_pct, alpha, tau = M.pinv_pid(torch.as_tensor(eta, device=cuda_device), torch.as_tensor(nu, device=cuda_device),
                                       torch.as_tensor(ref, device=cuda_device), integ_t, return_tau=True)
        wn, wa, wtau, want_integ = PO.pinv_pid(eta.astype(np.float64), nu.astype(np.float64), ref.astype(np.float64),
                                               want_integ)
        np.testing.assert_allclose(integ_t.cpu().numpy(), want_integ, rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(tau.cpu().numpy(), wtau, rtol=2e-6, atol=2e-4)
        # allocation parity is checked from the kernel's own (saturated, fp32) wrench
        wn2, wa2 = PO.allocate(tau.cpu().numpy().astype(np.float64))
        # n = sign(F) sqrt(|F| / K) amplifies fp32 rounding of F near zero (dn = dF / (2 K n)): compare the
        # physical force K n |n| everywhere and the percentage where the thruster is actually loaded.
        K = np.asarray(C.K_THRUST)[:, None]
        got = n_pct.cpu().numpy().astype(np.float64)
        np.testing.assert_allclose(K * got * np.abs(got), K * wn2 * np.abs(wn2), rtol=1e-5, atol=5e-5)
        loaded = np.abs(wn2) > 10.0
        np.testing.assert_allclose(got[loaded], wn2[loaded], rtol=2e-5, atol=0)
        big = np.hypot(*(np.linalg.pinv(PO.config_matrix()) @ tau.cpu().numpy().astype(np.float64))[0:2]) > 1e-3
        d = np.angle(np.exp(1j * (alpha.cpu().numpy() - wa2)))
        assert np.abs(d[0][big]).max() < 1e-5


def test_pinv_allocate_roundtrip(cuda_device):
    """Property at full size: B(alpha) F(n) reproduces tau wherever no thruster saturates."""
    import ml4ca_b200 as M
    n = 1 << 20
    g = torch.Generator(device=cuda_device); g.manual_seed(0)
    tau = (torch.rand(3, n, device=cuda_device, generator=g) * 2 - 1) * torch.tensor([[15.0], [8.0], [8.0]], device=cuda_device)
    n_pct, alpha = M.pinv_allocate(tau)
    K = torch.tensor(C.K_THRUST, device=cuda_device)[:, None]
    F = K * n_pct * n_pct.abs()
    lx, ly = C.LX, C.LY
    tx = F[0] * alpha[0].cos() + F[1] * alpha[1].cos()
    ty = F[0] * alpha[0].sin() + F[1] * alpha[1].sin() + F[2]
    tn = (F[0] * (lx[0] * alpha[0].sin() - ly[0] * alpha[0].cos()) + F[1] * (lx[1] * alpha[1].sin() - ly[1] * alpha[1].cos())
          + F[2] * lx[2])
    ok = (n_pct.abs() < 100.0).all(dim=0)
    assert float(ok.float().mean()) > 0.9
    err = torch.stack([tx, ty, tn]) - tau
    assert float(err[:, ok].abs().max()) < 2e-4
