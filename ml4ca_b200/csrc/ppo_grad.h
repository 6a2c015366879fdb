// ppo_grad.h -- argument block of one policy-gradient pass, shared by the host entry points (ppo_update.cu) and the three
// gradient kernels: ppo_grad_kernel (ppo_update.cu), ppo_grad_tc_kernel (ppo_update_tc.cu), ppo_grad_generic_kernel
// (ppo_update_generic.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ml4ca {

struct GradArgs {
  const float* params;     // flat fp32 master parameters (reference variable order)
  const __half* blob;      // packed fp16 operands of this net (tensor-core kernel: filled by its launcher)
  int obs, act, nout;      // nout = act (pi) or 1 (v)
  int hidden, n_hidden;    // H and NL: 64 x 64, 64^3, 80^3
  int off_w[4], off_b[4];  // flat offsets: [0] layer 1 (obs -> H), [l - 1] hidden layer l, [NL] output layer
  int off_ls;              // offset of pi/log_std
  int64_t n;               // envs (row length)
  int T;
  const float* obs_buf;    // [T, obs, n]
  const float* act_buf;    // [T, act, n]    (pi)
  const float* adv;        // [T, n]         (pi)
  const float* logp_old;   // [T, n]         (pi)
  const float* ret;        // [T, n]         (v)
  float clip;
  // TRPO (spinup/algos/tf1/trpo): loss_mode 1 = d_kl = mean KL(pi_theta || pi_old) (trpo/core.py:52-60,98) in place of the PPO
  // surrogate: act_buf then carries mu_old [T, act, n] and kl_ls_old the old log_std [act]; adv / logp_old unused.
  // mu_out [T, act, n] (nullable): forward only, the means of every sample are stored and no gradient is computed.
  int loss_mode;
  const float* kl_ls_old;
  float* mu_out;
  float* grad;             // flat, same layout as params; this net's block is accumulated into (caller zeroes)
  double* stats;           // [8]: 0 sum pi objective, 1 sum (ret - v)^2, 2 sum 0.5 (logp_old - logp)^2, 3 sum -logp,
                           //      4 clipped count, 5 sample count
  const int32_t* ctl;      // ml4ca_ppo_ctl (device) or NULL: skip the pass when ctl[0] != 0 && ctl[1] < iter
  int iter;
};

constexpr int kTcBlobHalves = 80 * 16 + 2 * 80 * 96 + 16 * 96 + 80 * 16 + 2 * 80 * 80;   // tensor-core operands of 80^3, the largest

}  // namespace ml4ca

// The launchers take a non-empty batch (n * T > 0).
int ml4ca_ppo_grad_generic_launch(const ml4ca::GradArgs& args, int activation, int net, cudaStream_t st);
// Shapes the tensor-core kernel is built for (64 x 64, 64^3, 80^3; obs_dim <= 15, act_dim <= 8).
bool ml4ca_ppo_tc_supports(int hidden, int n_hidden, int obs, int act);
// Packs the operands into `blob` (>= kTcBlobHalves halves of device scratch) and launches the kernel.
int ml4ca_ppo_grad_tc_launch(const ml4ca::GradArgs& args, int activation, int net, void* blob, cudaStream_t st);
