"""GPU parity of K1 (the batched thrust allocator, csrc/qp_alloc.cu + qp_slsqp.cuh) against the reference solver, ROW BY ROW.

The reference hands its NLP to SciPy's SLSQP (qp_allocator.py:206).  The kernel follows SLSQP's own path in float64, so
the comparison is literal: tests/golden/qp_config1.npz holds what QPTA.solve_QP itself returned on the 4096-demand
config-1 batch (BASELINE configs[0]), plus the reference run with a 1e-9 input perturbation and with exact derivatives,
which is what lets every non-literal row be explained (tests/qp_parity.py):
  1. success flags equal on all 4096 demands (hold-previous path taken on exactly the same demands);
  2. >= 99 % of the joint successes within 1e-5 max(1, |x|) of the reference's own output; every other row is either equal
     to the reference run with exact derivatives or a row where the reference does not reproduce itself to 1e-5 -- zero
     unexplained rows, no other-basin answers, the reference's active set on every row;
  3. the cleaned x (:232), the post-processing (hold on failure, F -> % thrust, mapToPi, bow gain, :267-320) and the
     objective switches (:108,116-150) against the reference's outputs;
  4. at the full benchmark size (1 Mi demands): the 4096-demand batch tiled 256 times gives 256 identical copies.
"""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, golden
from oracle import qp_oracle as QO

sys.path.insert(0, os.path.join(ROOT, "tests"))
import qp_parity  # noqa: E402

pytestmark = pytest.mark.gpu


def run_solver(dev, tau, prev, **kw):
    import ml4ca_b200 as M
    n = tau.shape[1]
    ta = M.QPTA(num_envs=n, device=dev)
    ta.previous_thruster_state = prev
    x, ok = ta.solve_QP(torch.as_tensor(tau, dtype=torch.float32, device=dev), **kw)
    st = ta.last_status.cpu().numpy().astype(np.uint32)
    return x.cpu().numpy().astype(np.float64), ok.cpu().numpy(), st


def test_row_by_row_against_the_reference(cuda_device):
    g = golden("qp_config1.npz")
    assert g['tau'].shape[1] == 4096
    x, ok, st = run_solver(cuda_device, g['tau'], g['prev'], raw=True)
    mask, it, mode = (st >> 1) & 0xFFFF, st >> 24, (st >> 17) & 15
    np.testing.assert_array_equal(ok, mode == 0)
    # the kernel returns fp32 rows: compare at fp32 resolution of the reference's numbers
    cls, dist = qp_parity.classify(g, x, ok, mask.astype(np.int32))
    counts = {k: int((cls == k).sum()) for k in ('A', 'B', 'C', 'FAIL', 'FLAG', 'X')}
    report = qp_parity.table(g, cls, dist, it, "K1 on the device vs QPTA.solve_QP, 4096 demands")
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        open(os.path.join(out, "qp_parity_gpu.md"), "w").write(report + "\n")
    assert counts['FLAG'] == 0 and counts['X'] == 0, report
    assert counts['A'] >= 0.99 * (counts['A'] + counts['B'] + counts['C']), counts
    assert counts['C'] <= 10, counts
    both = np.isin(cls, ['A', 'B', 'C'])
    np.testing.assert_array_equal(mask[both], g['mask_raw'][both].astype(np.uint32))
    assert (it[both] == g['slsqp_nit'][both]).mean() >= 0.98
    tail = slice(int(round(0.9 * 4096)), None)                  # grossly infeasible demands: the hold-previous path
    assert ok[tail].mean() < 0.1


def test_cleaned_output_and_callback_against_the_reference(cuda_device):
    import ml4ca_b200 as M
    g = golden("qp_config1.npz")
    n = g['tau'].shape[1]
    x, ok, st = run_solver(cuda_device, g['tau'], g['prev'])
    xr, okr, _ = run_solver(cuda_device, g['tau'], g['prev'], raw=True)
    np.testing.assert_array_equal(ok, g['success'])
    literal = ok & (qp_parity._rel(xr, g['x_raw']) <= 1e-5)
    # the |x| < 0.01 clean-up (:232): identical decisions wherever the raw value is not within 1e-5 of the threshold
    near = np.abs(np.abs(g['x_raw']) - 0.01) < 2e-5
    safe = literal & ~near.any(axis=0)
    np.testing.assert_array_equal(x[:, safe] == 0.0, g['x'][:, safe] == 0.0)
    np.testing.assert_allclose(x[:, safe], g['x'][:, safe], rtol=1e-5, atol=1e-5)
    # tau_controller_callback_func (:247-320)
    ta = M.QPTA(num_envs=n, device=cuda_device)
    ta.previous_thruster_state = g['prev']
    prev_before = ta.previous_thruster_state.clone()
    msg = ta.tau_controller_callback_func(torch.as_tensor(g['tau'], dtype=torch.float32, device=cuda_device))
    okc = msg['success'].cpu().numpy()
    np.testing.assert_array_equal(okc, g['success'])
    new_prev = ta.previous_thruster_state.cpu().numpy().astype(np.float64)
    out = ta.last_output.cpu().numpy().astype(np.float64)
    held = ~okc     # failed solves hold the previous state exactly (:267-269), angles through mapToPi (:277)
    np.testing.assert_array_equal(new_prev[:3, held], prev_before.cpu().numpy()[:3, held])
    np.testing.assert_allclose(new_prev[3:5, held], QO.map_to_pi(prev_before.cpu().numpy()[3:5, held].astype(np.float64)),
                               atol=1e-6)
    K = np.asarray(QO.C.K_THRUST)[:, None]
    F = new_prev[:3]
    np.testing.assert_allclose(out[:3], np.sign(F / K) * np.sqrt(np.abs(F / K)), rtol=2e-6, atol=1e-5)
    np.testing.assert_allclose(out[6], np.clip(2.5 * out[2], -100, 100), rtol=1e-6, atol=1e-5)
    assert np.all(out[3:5] >= -np.pi - 1e-6) and np.all(out[3:5] < np.pi + 1e-6)
    np.testing.assert_allclose(out[5], np.pi / 2, atol=1e-6)
    # the reference's published messages and its new previous state, on the literal rows
    np.testing.assert_allclose(new_prev[:5, safe], g['new_prev'][:5, safe], rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(msg['pod_angle_port'].cpu().numpy()[safe], g['pod_angle_deg'][0, safe], atol=2e-3)
    loaded = safe & (np.abs(g['stern_effort'][0]) > 5)
    np.testing.assert_allclose(msg['port_effort'].cpu().numpy()[loaded], g['stern_effort'][0, loaded], rtol=1e-4)
    np.testing.assert_allclose(msg['throttle_bow'].cpu().numpy()[safe], g['bow_throttle'][safe], rtol=1e-3, atol=2e-2)


@pytest.mark.parametrize("case", ["nofuel", "noflick", "noang", "bare", "weighted"])
def test_objective_switches(cuda_device, case):
    """solve_QP(tau_d, weight_matrix, reduce_fuel, reduce_flickering, reduce_angular) (:108,116-150) against the
    reference called with the same arguments."""
    g = golden("qp_switches.npz")
    kw = {"nofuel": dict(reduce_fuel=False), "noflick": dict(reduce_flickering=False), "noang": dict(reduce_angular=False),
          "bare": dict(reduce_fuel=False, reduce_flickering=False, reduce_angular=False),
          "weighted": dict(weight_matrix=np.diag([2.0, 1.0, 0.5, 1.0, 0.5, 2.0, 0.1, 0.4, 0.3, 0.2, 0.5]))}[case]
    x, ok, st = run_solver(cuda_device, g['tau'], g['prev'], raw=True, **kw)
    ref = g[case + '__success']
    np.testing.assert_array_equal(ok, ref)
    d_ref = qp_parity._rel(x, g[case + '__x_raw'])
    d_exact = qp_parity._rel(x, g[case + '__x_raw_exact'])
    both = ok & ref
    literal = d_ref[both] <= 1e-5
    explained = literal | ((d_exact[both] <= 1e-5) & g[case + '__success_exact'][both])
    assert literal.mean() >= 0.97, (case, literal.mean())
    assert d_ref[both].max() <= 1e-3, (case, d_ref[both].max())
    assert (~explained).sum() <= 2, (case, (~explained).sum())


def test_single_env_reference_call_shape(cuda_device):
    import ml4ca_b200 as M
    ta = M.QPTA(num_envs=1, device=cuda_device)
    x, ok = ta.solve_QP(np.array([[2.0, 1.0, 0.5]]).T)
    assert x.shape == (8,) and isinstance(ok, bool) and ok
    xs, oks, raw = QO.solve_stock(np.array([2.0, 1.0, 0.5]), np.zeros(5))
    assert oks and np.max(np.abs(x - xs)) < 2e-5
    x2, ok2 = ta.solve_QP(np.array([[40.0, -20.0, 30.0]]).T)     # far outside what the rate limits allow
    assert ok2 is False
    with pytest.raises(NotImplementedError):
        Q = np.eye(11)
        Q[0, 1] = Q[1, 0] = 0.1                                   # a non-diagonal weight matrix is not built
        ta.solve_QP(np.zeros((3, 1)), weight_matrix=Q)


def test_both_kernel_mappings_agree(cuda_device, tmp_path):
    """One thread per demand (default) and one demand over 8 lanes (ML4CA_QP_MAPPING=group, csrc/qp_group.cuh) are the same
    solver: equal flags and iteration counts, end points equal to fp32 output resolution."""
    import subprocess
    code = ("import numpy as np, torch, sys; sys.path.insert(0, %r); import ml4ca_b200 as M; "
            "g = np.load(%r); ta = M.QPTA(num_envs=4096); ta.previous_thruster_state = g['prev']; "
            "x, ok = ta.solve_QP(torch.as_tensor(g['tau'], dtype=torch.float32, device='cuda'), raw=True); "
            "np.savez(sys.argv[1], x=x.cpu().numpy(), st=ta.last_status.cpu().numpy())")
    outs = []
    for mapping in ("thread", "group"):
        path = str(tmp_path / ("qp_mapping_%s.npz" % mapping))
        env = dict(os.environ, ML4CA_QP_MAPPING=mapping)
        subprocess.run([sys.executable, "-c", code % (ROOT, os.path.join(ROOT, "tests", "golden", "qp_config1.npz")), path],
                       check=True, env=env, cwd=ROOT)
        outs.append(np.load(path))
    a, b = outs
    sa, sb = a['st'].astype(np.uint32), b['st'].astype(np.uint32)
    np.testing.assert_array_equal(sa & 1, sb & 1)
    same = ((sa & 1) == 1) & ((sa >> 24) == (sb >> 24))
    assert same.sum() >= 0.995 * (sa & 1).sum()
    np.testing.assert_allclose(b['x'][:, same], a['x'][:, same], rtol=0, atol=2e-6)


def test_full_size_batch_is_the_tiled_small_one(cuda_device):
    """BASELINE's bench size (1 Mi demands): 256 copies of the 4096-demand golden batch must give 256 identical result
    blocks -- chunking, work fetching and indexing do not depend on the batch size."""
    g = golden("qp_config1.npz")
    reps = 256
    tau, prev = np.tile(g['tau'], (1, reps)), np.tile(g['prev'], (1, reps))
    x, ok, st = run_solver(cuda_device, tau, prev, raw=True)
    x0, ok0, st0 = run_solver(cuda_device, g['tau'], g['prev'], raw=True)
    np.testing.assert_array_equal(x.reshape(8, reps, 4096), np.broadcast_to(x0[:, None, :], (8, reps, 4096)))
    np.testing.assert_array_equal(st.reshape(reps, 4096), np.broadcast_to(st0[None, :], (reps, 4096)))
