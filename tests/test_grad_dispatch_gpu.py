"""Which gradient kernel each pass of csrc/ppo_update.cu runs, read from the kernel names torch.profiler records.
ml4ca_ppo_grad runs on the tensor cores unless ml4ca_ppo_use_fp32 is on; ml4ca_trpo_policy_mu and ml4ca_trpo_kl_grad run on them
only when ml4ca_trpo_use_tensor_cores is on.  Otherwise the fp32 kernel: ppo_grad_kernel for the 64 x 64 network with
obs_dim <= 12, ppo_grad_generic_kernel for every other network."""
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

pytestmark = pytest.mark.gpu

KERNELS = ("ppo_grad_kernel", "ppo_grad_tc_kernel", "ppo_grad_generic_kernel")


def _kernels_of(run):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    return sorted({k for k in KERNELS if any("::%s<" % k in name for name in names)})


@pytest.mark.parametrize("hidden,obs_dim", [((64, 64), 9), ((64, 64), 13), ((64, 64, 64), 9), ((80, 80, 80), 9)])
def test_each_pass_runs_the_kernel_its_switch_selects(cuda_device, hidden, obs_dim):
    import ml4ca_b200 as M
    from ml4ca_b200 import _lib
    L, P, st = _lib.lib(), _lib.ptr, _lib.current_stream()
    act_dim, T, n = 7, 2, 1000
    ac = M.ActorCritic(obs_dim, act_dim, hidden, "leaky_relu", device=cuda_device, seed=1)
    obs = torch.randn(T, obs_dim, n, device=cuda_device)
    act = torch.randn(T, act_dim, n, device=cuda_device)         # actions (PPO) or mu_old (TRPO KL)
    row = torch.randn(T, n, device=cuda_device)                  # adv, ret, logp_old
    log_std_old = torch.zeros(act_dim, device=cuda_device)
    mu = torch.empty(T, act_dim, n, device=cuda_device)
    grad = torch.empty(ac.num_params, device=cuda_device)
    stats = torch.empty(8, dtype=torch.float64, device=cuda_device)
    passes = {
        "ml4ca_ppo_grad pi": lambda: L.ml4ca_ppo_grad(ac._handle, 0, n, T, P(obs), P(act), P(row), P(row), P(row), 0.2, P(grad),
                                                      P(stats), st),
        "ml4ca_ppo_grad v": lambda: L.ml4ca_ppo_grad(ac._handle, 1, n, T, P(obs), P(act), P(row), P(row), P(row), 0.2, P(grad),
                                                     P(stats), st),
        "ml4ca_trpo_policy_mu": lambda: L.ml4ca_trpo_policy_mu(ac._handle, n, T, P(obs), P(mu), st),
        "ml4ca_trpo_kl_grad": lambda: L.ml4ca_trpo_kl_grad(ac._handle, n, T, P(obs), P(act), P(log_std_old), P(grad), P(stats), st),
    }
    fp32_kernel = "ppo_grad_kernel" if hidden == (64, 64) and obs_dim <= 12 else "ppo_grad_generic_kernel"
    prev = L.ml4ca_ppo_use_fp32(-1), L.ml4ca_trpo_use_tensor_cores(-1)
    try:
        for use_fp32 in (0, 1):
            for trpo_tc in (0, 1):
                L.ml4ca_ppo_use_fp32(use_fp32)
                L.ml4ca_trpo_use_tensor_cores(trpo_tc)
                for name, call in passes.items():
                    tensor_cores = not use_fp32 if name.startswith("ml4ca_ppo_grad") else bool(trpo_tc)
                    want = "ppo_grad_tc_kernel" if tensor_cores else fp32_kernel
                    ran = _kernels_of(lambda: _lib.check(call(), name))
                    assert ran == [want], (name, dict(use_fp32=use_fp32, trpo_tc=trpo_tc), ran)
    finally:
        L.ml4ca_ppo_use_fp32(prev[0])
        L.ml4ca_trpo_use_tensor_cores(prev[1])
