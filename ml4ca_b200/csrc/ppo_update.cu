// ppo_update.cu -- K6: PPO policy / value gradients over the whole trajectory buffer, and the Adam step.
//
// Replaces the TensorFlow graph pieces of /root/reference/src/rl/windows_workspace/spinup/algos/tf1/ppo/ppo.py:
//   :234-237  ratio = exp(logp - logp_old);  min_adv = where(adv > 0, (1 + c) adv, (1 - c) adv)
//             pi_loss = -mean(min(ratio adv, min_adv));  v_loss = mean((ret - v)^2)
//   :241-245  approx_kl = 0.5 mean((logp_old - logp)^2), approx_ent = mean(-logp), clipfrac
//   :249-250  train_pi / train_v = MpiAdamOptimizer(lr).minimize(loss)   (spinup/utils/mpi_tf.py:45-80)
// with logp from core.gaussian_likelihood (core.py:42-46) and the networks of core.mlp (core.py:29-33).
//
// ppo_grad_kernel<ACTIVATION, NET>: forward, loss and backward of ONE network (NET 0 = pi incl. log_std, 1 = v) for
// every sample of a [T, ., n] buffer, in fp32.  A CTA works on tiles of 128 samples:
//   global rows -> smem (feature-major rows of 128 samples, stride 132: conflict-free 128-bit accesses)
//   H1 = f(X0 W1 + b1), H2 = f(H1 W2 + b2), OUT = H2 Wo + bo         register-tiled GEMMs, 8 samples x 4 features / thread
//   per-sample loss -> dOUT (sum convention: the caller divides by the global sample count)
//   dWo += H2^T dOUT,  G = (dOUT Wo^T) .* f'(H2),  dW2 += H1^T G,  G = (G W2^T) .* f'(H1),  dW1 += X0^T G  (+ bias sums)
// Weight-gradient accumulators live in registers across all tiles of the CTA (persistent grid = one CTA per SM) and
// are flushed once with atomicAdd; loss statistics accumulate in double.  A thread's four features are
// {tx, tx + 16, tx + 32, tx + 48}: consecutive lanes then touch consecutive smem rows, and the weight copies in
// shared memory are stored column-permuted so that those four weights are one 128-bit load.
//
// Bound: FP32 FMA pipe (~15.6 k FMA per sample and network against 77 B of HBM traffic).  This is the CUDA-core
// version; moving the three big GEMMs per layer onto tcgen05 (MN-major views of the same smem operands) is
// round-2 work (DESIGN.md section 3).
//
// Host side: every gradient entry point (PPO, TRPO KL, TRPO forward-only) fills one GradArgs (ppo_grad.h) and goes through
// grad_pass, which picks this kernel, the tcgen05 one (ppo_update_tc.cu) or the generic fp32 one (ppo_update_generic.cu) for
// the networks ml4ca_policy_create accepts: 64 x 64, 64^3 and 80^3.
#include <new>

#include <stdlib.h>

#include "common.h"
#include "ppo_grad.h"

namespace ml4ca {
namespace ppo {

constexpr int TS = 128;   // samples per tile
constexpr int RS = 132;   // smem row stride in floats
constexpr int H = 64;     // hidden width (BASELINE config 64 x 64)
constexpr int OP = 8;     // padded output width (act_dim <= 7, value head 1)
constexpr int XR = 12;    // padded input rows (obs_dim <= 12)

// the device-side early stop of the policy loop (include/ml4ca_b200.h: ml4ca_ppo_ctl)
__device__ __forceinline__ bool pass_skipped(const int32_t* ctl, int iter) {
  return ctl != nullptr && ctl[0] != 0 && ctl[1] < iter;
}

struct Smem {
  float w1p[XR][H];     // w1p[k][4 tx + b] = W1[k][tx + 16 b]
  float w2p[H][H];      // w2p[k][4 tx + b] = W2[k][tx + 16 b]
  float w2tp[H][H];     // w2tp[j][4 tx + b] = W2[tx + 16 b][j]
  float wo[H][OP];      // wo[k][o]
  float wotp[OP][H];    // wotp[o][4 tx + b] = Wo[tx + 16 b][o]
  float b1[H], b2[H], bo[OP];
  float sd[OP], inv[OP], ls[OP];   // exp(log_std), 1 / (exp(log_std) + 1e-8), log_std
  float kiv[OP], kls[OP];          // KL mode: 1 / (exp(2 log_std_old) + 1e-8), log_std_old
  float x0[XR][RS];
  float h1[H][RS];
  float h2[H][RS];
  float g[H][RS];
  float out[OP][RS];    // OUT, then dOUT in place
  float actb[OP][RS];   // actions taken (pi)
  float aux0[RS];       // adv (pi) / ret (v)
  float aux1[RS];       // logp_old (pi)
  double red[8][8];     // per-warp partial statistics
};

template <int ACTIVATION>
__device__ __forceinline__ float act_fn(float z) {
  if constexpr (ACTIVATION == 1) return fmaxf(z, 0.2f * z);   // tf.nn.leaky_relu, alpha = 0.2
  return tanhf(z);
}
template <int ACTIVATION>
__device__ __forceinline__ float act_grad(float h) {          // derivative expressed through the OUTPUT h = f(z)
  if constexpr (ACTIVATION == 1) return h > 0.f ? 1.0f : 0.2f;
  return 1.0f - h * h;
}

__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// acc[i][b] (+)= sum_k in[k][8 ty + i] * wp[k][4 tx + b]   for k < K
template <int WSTRIDE>
__device__ __forceinline__ void gemm_tile(float (&acc)[8][4], const float (*in)[RS], const float* wp, int K, int tx, int ty) {
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    const float4 a0 = lds4(&in[k][8 * ty]), a1 = lds4(&in[k][8 * ty + 4]);
    const float4 w = lds4(wp + k * WSTRIDE + 4 * tx);
    const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[i][b] = fmaf(a[i], ww[b], acc[i][b]);
  }
}

template <int ACTIVATION, int NET>
__global__ void __launch_bounds__(256, 1) ppo_grad_kernel(const GradArgs A) {
  if (pass_skipped(A.ctl, A.iter)) return;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  Smem& S = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int obs = A.obs, nout = A.nout;

  // ---- weights -> smem (column-permuted copies, see header) -----------------------------------------------------------
  for (int e = tid; e < XR * H; e += 256) {
    const int k = e / H, c = e % H, f = (c >> 2) + 16 * (c & 3);
    S.w1p[k][c] = k < obs ? A.params[A.off_w[0] + k * H + f] : 0.f;
  }
  for (int e = tid; e < H * H; e += 256) {
    const int r = e / H, c = e % H, f = (c >> 2) + 16 * (c & 3);
    S.w2p[r][c] = A.params[A.off_w[1] + r * H + f];      // W2[k = r][j = f]
    S.w2tp[r][c] = A.params[A.off_w[1] + f * H + r];     // W2[k = f][j = r]
  }
  for (int e = tid; e < H * OP; e += 256) {
    const int k = e / OP, o = e % OP;
    S.wo[k][o] = o < nout ? A.params[A.off_w[2] + k * nout + o] : 0.f;
  }
  for (int e = tid; e < OP * H; e += 256) {
    const int o = e / H, c = e % H, f = (c >> 2) + 16 * (c & 3);
    S.wotp[o][c] = o < nout ? A.params[A.off_w[2] + f * nout + o] : 0.f;
  }
  if (tid < H) S.b1[tid] = A.params[A.off_b[0] + tid], S.b2[tid] = A.params[A.off_b[1] + tid];
  if (tid < OP) {
    S.bo[tid] = tid < nout ? A.params[A.off_b[2] + tid] : 0.f;
    const float ls = (NET == 0 && tid < nout) ? A.params[A.off_ls + tid] : 0.f;
    const float sd = expf(ls);
    S.ls[tid] = ls, S.sd[tid] = sd, S.inv[tid] = 1.0f / (sd + 1e-8f);
    const float lo = (NET == 0 && A.loss_mode == 1 && tid < nout) ? A.kl_ls_old[tid] : 0.f;
    S.kls[tid] = lo, S.kiv[tid] = 1.0f / (expf(2.0f * lo) + 1e-8f);               // trpo/core.py:57-58
  }
  // zero the padding rows / columns once
  for (int e = tid; e < XR * RS; e += 256) (&S.x0[0][0])[e] = 0.f;
  for (int e = tid; e < OP * RS; e += 256) (&S.actb[0][0])[e] = 0.f, (&S.out[0][0])[e] = 0.f;

  // ---- persistent accumulators ------------------------------------------------------------------------------------------
  float dW2[4][4];      // rows k = 4 tk + a (tk = ty), columns j = tx + 16 b
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) dW2[a][b] = 0.f;
  float dWo[2] = {0.f, 0.f};        // row k = tid >> 2, outputs o = 2 (tid & 3), +1
  float dW1[3] = {0.f, 0.f, 0.f};   // column j = tid & 63, rows k = (tid >> 6) + 4 m
  float db1 = 0.f, db2 = 0.f;       // feature tid >> 2 (valid in lanes with (tid & 3) == 0)
  float dbo = 0.f;                  // output tid >> 5 for tid < 256: warp w sums output w
  float dls_a[OP];                 // thread = sample: sum over its samples of dL/dlog_std[a]
#pragma unroll
  for (int o = 0; o < OP; ++o) dls_a[o] = 0.f;
  double st[5] = {0.0, 0.0, 0.0, 0.0, 0.0};

  const int64_t n = A.n;
  const int64_t total = n * (int64_t)A.T;       // tiles run over the flat sample index (common.h: split_sample)
  const int64_t num_tiles = (total + TS - 1) / TS;
  const int rows_in = obs + (NET == 0 ? A.act + 2 : 1);   // obs rows, then (pi) act rows, adv, logp_old | (v) ret
  constexpr int kLoads = (XR + OP + 2) * TS / 256;         // 11 >= rows_in * 128 / 256
  float pre[kLoads];

  auto fetch = [&](int64_t tile) {
    const int64_t smp = tile * TS + (tid & 127);   // the column of every load of this thread (256 % 128 == 0)
    const bool live = smp < total;
    int64_t t = 0, i = 0;
    if (live) split_sample(smp, n, t, i);
#pragma unroll
    for (int m = 0; m < kLoads; ++m) {
      const int idx = tid + 256 * m, row = idx >> 7;
      float v = 0.f;
      if (row < rows_in && live) {
        const float* base;     // rows a mode does not use have a NULL base and read as zero
        int64_t off;
        if (row < obs) base = A.obs_buf, off = ((int64_t)t * obs + row) * n;
        else if (NET == 1) base = A.ret, off = (int64_t)t * n;
        else if (row < obs + A.act) base = A.act_buf, off = ((int64_t)t * A.act + (row - obs)) * n;
        else if (row == obs + A.act) base = A.adv, off = (int64_t)t * n;
        else base = A.logp_old, off = (int64_t)t * n;
        if (base != nullptr) v = __ldg(base + off + i);
      }
      pre[m] = v;
    }
  };
  auto stash = [&]() {
#pragma unroll
    for (int m = 0; m < kLoads; ++m) {
      const int idx = tid + 256 * m, row = idx >> 7, col = idx & 127;
      if (row >= rows_in) continue;
      if (row < obs) S.x0[row][col] = pre[m];
      else if (NET == 1) S.aux0[col] = pre[m];
      else if (row < obs + A.act) S.actb[row - obs][col] = pre[m];
      else if (row == obs + A.act) S.aux0[col] = pre[m];
      else S.aux1[col] = pre[m];
    }
  };

  int64_t tile = blockIdx.x;
  if (tile < num_tiles) fetch(tile);
  __syncthreads();

  for (; tile < num_tiles; tile += gridDim.x) {
    const int valid = (int)((total - tile * TS) < TS ? (total - tile * TS) : TS);
    stash();
    __syncthreads();
    if (tile + gridDim.x < num_tiles) fetch(tile + gridDim.x);   // next tile's rows travel while this one computes

    float acc[8][4];
    // ---- 1. H1 = f(X0 W1 + b1) ------------------------------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[i][b] = S.b1[tx + 16 * b];
    gemm_tile<H>(acc, S.x0, &S.w1p[0][0], obs, tx, ty);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      float4 lo = make_float4(act_fn<ACTIVATION>(acc[0][b]), act_fn<ACTIVATION>(acc[1][b]), act_fn<ACTIVATION>(acc[2][b]), act_fn<ACTIVATION>(acc[3][b]));
      float4 hi = make_float4(act_fn<ACTIVATION>(acc[4][b]), act_fn<ACTIVATION>(acc[5][b]), act_fn<ACTIVATION>(acc[6][b]), act_fn<ACTIVATION>(acc[7][b]));
      *reinterpret_cast<float4*>(&S.h1[tx + 16 * b][8 * ty]) = lo;
      *reinterpret_cast<float4*>(&S.h1[tx + 16 * b][8 * ty + 4]) = hi;
    }
    __syncthreads();
    // ---- 2. H2 = f(H1 W2 + b2) ------------------------------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[i][b] = S.b2[tx + 16 * b];
    gemm_tile<H>(acc, S.h1, &S.w2p[0][0], H, tx, ty);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      float4 lo = make_float4(act_fn<ACTIVATION>(acc[0][b]), act_fn<ACTIVATION>(acc[1][b]), act_fn<ACTIVATION>(acc[2][b]), act_fn<ACTIVATION>(acc[3][b]));
      float4 hi = make_float4(act_fn<ACTIVATION>(acc[4][b]), act_fn<ACTIVATION>(acc[5][b]), act_fn<ACTIVATION>(acc[6][b]), act_fn<ACTIVATION>(acc[7][b]));
      *reinterpret_cast<float4*>(&S.h2[tx + 16 * b][8 * ty]) = lo;
      *reinterpret_cast<float4*>(&S.h2[tx + 16 * b][8 * ty + 4]) = hi;
    }
    __syncthreads();
    // ---- 3. OUT = H2 Wo + bo : thread = (sample tid & 127, output half tid >> 7) ---------------------------------------
    {
      const int s = tid & 127, half = tid >> 7;
      float o4[4] = {S.bo[4 * half], S.bo[4 * half + 1], S.bo[4 * half + 2], S.bo[4 * half + 3]};
#pragma unroll 8
      for (int k = 0; k < H; ++k) {
        const float a = S.h2[k][s];
        const float4 w = lds4(&S.wo[k][4 * half]);
        o4[0] = fmaf(a, w.x, o4[0]), o4[1] = fmaf(a, w.y, o4[1]), o4[2] = fmaf(a, w.z, o4[2]), o4[3] = fmaf(a, w.w, o4[3]);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) S.out[4 * half + q][s] = o4[q];
    }
    __syncthreads();
    if (A.mu_out != nullptr) {   // forward only (uniform branch): store the means, next tile
      if (tid < TS && tid < valid) {
        int64_t t, i;
        split_sample(tile * TS + tid, n, t, i);
        for (int a = 0; a < nout; ++a) A.mu_out[((int64_t)t * nout + a) * n + i] = S.out[a][tid];
      }
      __syncthreads();           // the next tile overwrites x0 / out
      continue;
    }
    // ---- 4. loss and dOUT (sum convention), one thread per sample -------------------------------------------------------
    if (tid < TS) {
      const int s = tid;
      const bool live = s < valid;
      if (NET == 0 && A.loss_mode == 1) {
        // d_kl = mean_s sum_a 0.5 (((mu_old - mu)^2 + var) / (var_old + EPS) - 1) + log_std_old - log_std   (trpo/core.py:52-60
        // with mu0 = the current policy, mu1 = the old one, as mlp_gaussian_policy calls it, :98)
        double kl = 0.0;
#pragma unroll
        for (int a = 0; a < OP; ++a) {
          if (a < nout) {
            const float d = S.out[a][s] - S.actb[a][s], var = S.sd[a] * S.sd[a];
            kl += (double)(0.5f * ((d * d + var) * S.kiv[a] - 1.0f) + (S.kls[a] - S.ls[a]));
            S.out[a][s] = live ? d * S.kiv[a] : 0.f;                               // d kl / d mu
            dls_a[a] += live ? (var * S.kiv[a] - 1.0f) : 0.f;                      // d kl / d log_std
          } else {
            S.out[a][s] = 0.f;
          }
        }
        if (live) st[2] += kl;
      } else if constexpr (NET == 0) {
        float logp = 0.f, z[OP], dmu[OP];
#pragma unroll
        for (int a = 0; a < OP; ++a) {
          z[a] = 0.f, dmu[a] = 0.f;
          if (a < nout) {
            z[a] = (S.actb[a][s] - S.out[a][s]) * S.inv[a];                       // (x - mu) / (exp(log_std) + EPS), core.py:45
            logp += -0.5f * (z[a] * z[a] + 2.0f * S.ls[a] + 1.8378770664093453f);
          }
        }
        const float adv = S.aux0[s], lpo = S.aux1[s];
        const float ratio = expf(logp - lpo);                                      // ppo.py:234
        const float min_adv = adv > 0.f ? (1.0f + A.clip) * adv : (1.0f - A.clip) * adv;   // :235
        const float ra = ratio * adv;
        const bool use_ratio = ra <= min_adv;                                      // tf.minimum sends the gradient to x where x <= y
        const float dlogp = (live && use_ratio) ? -ra : 0.f;                       // d(-min(ratio adv, min_adv)) / dlogp
#pragma unroll
        for (int a = 0; a < OP; ++a) {
          if (a < nout) {
            S.out[a][s] = dlogp * z[a] * S.inv[a];                                 // dlogp/dmu = (x - mu) / (std + EPS)^2
            dls_a[a] += dlogp * (z[a] * z[a] * S.sd[a] * S.inv[a] - 1.0f);         // dlogp/dlog_std = z^2 std / (std + EPS) - 1
          } else {
            S.out[a][s] = 0.f;
          }
        }
        if (live) {
          st[0] += (double)fminf(ra, min_adv);
          const float dl = lpo - logp;
          st[2] += 0.5 * (double)dl * (double)dl;                                  // :242
          st[3] += (double)(-logp);                                                // :243
          st[4] += (ratio > 1.0f + A.clip || ratio < 1.0f - A.clip) ? 1.0 : 0.0;   // :244
        }
      } else {
        const float v = S.out[0][s], r = S.aux0[s];
        const float e = v - r;
        S.out[0][s] = live ? 2.0f * e : 0.f;                                       // d(ret - v)^2 / dv
#pragma unroll
        for (int a = 1; a < OP; ++a) S.out[a][s] = 0.f;
        if (live) st[1] += (double)e * (double)e;                                  // :236
      }
    }
    __syncthreads();
    // ---- 5. dWo += H2^T dOUT ; dbo ----------------------------------------------------------------------------------------
    {
      const int k = tid >> 2, o = 2 * (tid & 3);
      float s0 = 0.f, s1 = 0.f;
#pragma unroll 4
      for (int s = 0; s < TS; s += 4) {
        const float4 h = lds4(&S.h2[k][s]), d0 = lds4(&S.out[o][s]), d1 = lds4(&S.out[o + 1][s]);
        s0 += h.x * d0.x + h.y * d0.y + h.z * d0.z + h.w * d0.w;
        s1 += h.x * d1.x + h.y * d1.y + h.z * d1.z + h.w * d1.w;
      }
      dWo[0] += s0, dWo[1] += s1;
      const int w = tid >> 5, lane = tid & 31;     // warp w sums dOUT row w
      const float4 d = lds4(&S.out[w][4 * lane]);
      float r = d.x + d.y + d.z + d.w;
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, off);
      dbo += r;
    }
    // ---- 6. G = (dOUT Wo^T) .* f'(H2) ---------------------------------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[i][b] = 0.f;
    gemm_tile<H>(acc, S.out, &S.wotp[0][0], OP, tx, ty);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const float4 h0 = lds4(&S.h2[tx + 16 * b][8 * ty]), h1v = lds4(&S.h2[tx + 16 * b][8 * ty + 4]);
      float4 lo = make_float4(acc[0][b] * act_grad<ACTIVATION>(h0.x), acc[1][b] * act_grad<ACTIVATION>(h0.y),
                              acc[2][b] * act_grad<ACTIVATION>(h0.z), acc[3][b] * act_grad<ACTIVATION>(h0.w));
      float4 hi = make_float4(acc[4][b] * act_grad<ACTIVATION>(h1v.x), acc[5][b] * act_grad<ACTIVATION>(h1v.y),
                              acc[6][b] * act_grad<ACTIVATION>(h1v.z), acc[7][b] * act_grad<ACTIVATION>(h1v.w));
      *reinterpret_cast<float4*>(&S.g[tx + 16 * b][8 * ty]) = lo;
      *reinterpret_cast<float4*>(&S.g[tx + 16 * b][8 * ty + 4]) = hi;
    }
    __syncthreads();
    // ---- 7. dW2 += H1^T G ; db2 ---------------------------------------------------------------------------------------------
    {
#pragma unroll 2
      for (int s = 0; s < TS; s += 4) {
        float4 hk[4], gj[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) hk[a] = lds4(&S.h1[4 * ty + a][s]);
#pragma unroll
        for (int b = 0; b < 4; ++b) gj[b] = lds4(&S.g[tx + 16 * b][s]);
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b)
            dW2[a][b] += hk[a].x * gj[b].x + hk[a].y * gj[b].y + hk[a].z * gj[b].z + hk[a].w * gj[b].w;
      }
      const int j = tid >> 2, q = tid & 3;
      float r = 0.f;
#pragma unroll
      for (int s = 0; s < 32; s += 4) {
        const float4 d = lds4(&S.g[j][32 * q + s]);
        r += d.x + d.y + d.z + d.w;
      }
      r += __shfl_xor_sync(0xFFFFFFFFu, r, 1);
      r += __shfl_xor_sync(0xFFFFFFFFu, r, 2);
      db2 += r;
    }
    // ---- 8. G = (G W2^T) .* f'(H1) --------------------------------------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[i][b] = 0.f;
    gemm_tile<H>(acc, S.g, &S.w2tp[0][0], H, tx, ty);
    __syncthreads();   // every thread has finished reading G
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const float4 h0 = lds4(&S.h1[tx + 16 * b][8 * ty]), h1v = lds4(&S.h1[tx + 16 * b][8 * ty + 4]);
      float4 lo = make_float4(acc[0][b] * act_grad<ACTIVATION>(h0.x), acc[1][b] * act_grad<ACTIVATION>(h0.y),
                              acc[2][b] * act_grad<ACTIVATION>(h0.z), acc[3][b] * act_grad<ACTIVATION>(h0.w));
      float4 hi = make_float4(acc[4][b] * act_grad<ACTIVATION>(h1v.x), acc[5][b] * act_grad<ACTIVATION>(h1v.y),
                              acc[6][b] * act_grad<ACTIVATION>(h1v.z), acc[7][b] * act_grad<ACTIVATION>(h1v.w));
      *reinterpret_cast<float4*>(&S.g[tx + 16 * b][8 * ty]) = lo;
      *reinterpret_cast<float4*>(&S.g[tx + 16 * b][8 * ty + 4]) = hi;
    }
    __syncthreads();
    // ---- 9. dW1 += X0^T G ; db1 -----------------------------------------------------------------------------------------------
    {
      const int j = tid & 63, kq = tid >> 6;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll 4
      for (int s = 0; s < TS; s += 4) {
        const float4 gj = lds4(&S.g[j][s]);
        const float4 x0 = lds4(&S.x0[kq][s]), x1 = lds4(&S.x0[kq + 4][s]), x2 = lds4(&S.x0[kq + 8][s]);
        s0 += x0.x * gj.x + x0.y * gj.y + x0.z * gj.z + x0.w * gj.w;
        s1 += x1.x * gj.x + x1.y * gj.y + x1.z * gj.z + x1.w * gj.w;
        s2 += x2.x * gj.x + x2.y * gj.y + x2.z * gj.z + x2.w * gj.w;
      }
      dW1[0] += s0, dW1[1] += s1, dW1[2] += s2;
      const int jj = tid >> 2, q = tid & 3;
      float r = 0.f;
#pragma unroll
      for (int s = 0; s < 32; s += 4) {
        const float4 d = lds4(&S.g[jj][32 * q + s]);
        r += d.x + d.y + d.z + d.w;
      }
      r += __shfl_xor_sync(0xFFFFFFFFu, r, 1);
      r += __shfl_xor_sync(0xFFFFFFFFu, r, 2);
      db1 += r;
    }
    __syncthreads();   // the next tile overwrites x0 / actb / aux
  }

  if (A.mu_out != nullptr) return;   // forward-only pass (uniform)
  // ---- flush: one atomicAdd per accumulator and CTA ------------------------------------------------------------------------------
  float* g = A.grad;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) atomicAdd(g + A.off_w[1] + (4 * ty + a) * H + (tx + 16 * b), dW2[a][b]);
  {
    const int k = tid >> 2, o = 2 * (tid & 3);
    if (o < nout) atomicAdd(g + A.off_w[2] + k * nout + o, dWo[0]);
    if (o + 1 < nout) atomicAdd(g + A.off_w[2] + k * nout + o + 1, dWo[1]);
    const int j = tid & 63, kq = tid >> 6;
    if (kq < obs) atomicAdd(g + A.off_w[0] + kq * H + j, dW1[0]);
    if (kq + 4 < obs) atomicAdd(g + A.off_w[0] + (kq + 4) * H + j, dW1[1]);
    if (kq + 8 < obs) atomicAdd(g + A.off_w[0] + (kq + 8) * H + j, dW1[2]);
    if ((tid & 3) == 0) {
      atomicAdd(g + A.off_b[0] + (tid >> 2), db1);
      atomicAdd(g + A.off_b[1] + (tid >> 2), db2);
    }
    const int w = tid >> 5;
    if ((tid & 31) == 0 && w < nout) atomicAdd(g + A.off_b[2] + w, dbo);
  }
  // log_std gradient and statistics: reduce over the 128 sample threads (warps 0-3)
  if (tid < TS) {
#pragma unroll
    for (int a = 0; a < OP; ++a) {
      float r = dls_a[a];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, off);
      if (NET == 0 && (tid & 31) == 0 && a < nout) atomicAdd(g + A.off_ls + a, r);
    }
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      double r = st[q];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, off);
      if ((tid & 31) == 0) S.red[tid >> 5][q] = r;
    }
  }
  __syncthreads();
  if (tid < 5) {
    const double r = S.red[0][tid] + S.red[1][tid] + S.red[2][tid] + S.red[3][tid];
    if (r != 0.0) atomicAdd(A.stats + tid, r);
  }
  if (tid == 0 && blockIdx.x == 0) atomicAdd(A.stats + 5, (double)A.n * (double)A.T);
}

// TF-1 Adam (tf.train.AdamOptimizer defaults beta1 0.9, beta2 0.999, eps 1e-8; mpi_tf.py:45):
//   lr_t = lr sqrt(1 - beta2^t) / (1 - beta1^t);  m <- b1 m + (1 - b1) g;  v <- b2 v + (1 - b2) g^2;  p <- p - lr_t m / (sqrt(v) + eps)
__global__ void __launch_bounds__(256) adam_kernel(int64_t m, float* __restrict__ p, const float* __restrict__ grad,
                                                   float* __restrict__ m1, float* __restrict__ m2, float lr_t, float b1,
                                                   float b2, float eps, float gscale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  adam_update(p[i], m1[i], m2[i], __fmul_rn(grad[i], gscale), lr_t, b1, b2, eps);
}

// Adam step of one optimizer inside the update graph: step count and early stop come from the control block.
__global__ void __launch_bounds__(256) adam_dev_kernel(int64_t m, float* __restrict__ p, const float* __restrict__ grad,
                                                       float* __restrict__ m1, float* __restrict__ m2, float lr, float b1, float b2,
                                                       float eps, float gscale, int net, int iter,
                                                       const float* __restrict__ tail, float count, float kl_limit,
                                                       ml4ca_ppo_ctl* __restrict__ ctl) {
  const int32_t* c32 = reinterpret_cast<const int32_t*>(ctl);
  if (net == 0 && pass_skipped(c32, iter)) return;
  __shared__ float lr_t_s;
  if (threadIdx.x == 0) {
    const int t = (net == 0 ? ctl->t_pi : ctl->t_v) + iter + 1;
    lr_t_s = (float)((double)lr * sqrt(1.0 - pow((double)b2, (double)t)) / (1.0 - pow((double)b1, (double)t)));
  }
  __syncthreads();
  const float lr_t = lr_t_s;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) {
    adam_update(p[i], m1[i], m2[i], __fmul_rn(grad[i], gscale), lr_t, b1, b2, eps);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (iter == 0) {
      if (net == 0) {
        for (int q = 0; q < 5; ++q) ctl->first[q] = tail[q];
      } else {
        ctl->first[5] = tail[1];
      }
    }
    if (net == 0 && kl_limit > 0.f && tail[2] / count > kl_limit) {     // ppo.py:269-271; the step above stays applied
      ctl->stop_iter = iter;
      __threadfence();
      ctl->stop = 1;
    }
  }
}

__global__ void ppo_ctl_kernel(ml4ca_ppo_ctl* ctl, int begin, int pi_iters, int v_iters) {
  if (begin) {
    ctl->stop = 0, ctl->stop_iter = 0x7fffffff;
  } else {
    if (!ctl->stop) ctl->stop_iter = pi_iters - 1;
    ctl->t_pi += ctl->stop_iter + 1;
    ctl->t_v += v_iters;
  }
}

}  // namespace ppo
}  // namespace ml4ca

using namespace ml4ca;

static bool g_use_fp32 = [] {
  const char* e = getenv("ML4CA_PPO_FP32");
  return e != nullptr && atoi(e) != 0;
}();

extern "C" int ml4ca_ppo_use_fp32(int enable) {
  const int prev = g_use_fp32 ? 1 : 0;
  if (enable >= 0) g_use_fp32 = enable != 0;
  return prev;
}

static bool g_trpo_tc = false;   // TRPO passes on the tensor-core kernel (ml4ca_trpo_use_tensor_cores)

extern "C" int ml4ca_trpo_use_tensor_cores(int enable) {
  const int prev = g_trpo_tc ? 1 : 0;
  if (enable >= 0) g_trpo_tc = enable != 0;
  return prev;
}

// per-device scratch for the packed fp16 operands of the tensor-core gradient kernel (kept for the life of the process)
static int tc_blob(int32_t device, __half** out) {
  static __half* blob[64] = {};
  ML4CA_REQUIRE(device >= 0 && device < 64, "device index out of range");
  if (blob[device] == nullptr) ML4CA_CUDA(cudaMalloc(&blob[device], sizeof(__half) * kTcBlobHalves));
  *out = blob[device];
  return ML4CA_OK;
}

// policy.cu
extern "C" int ml4ca_policy_describe(const ml4ca_policy* p, ml4ca_policy_cfg* cfg, int32_t* device);

// Shape and flat offsets of net 0 (pi, then log_std) or net 1 (v) of a policy with configuration cfg.  A net's block is W1 [obs, H],
// b1, then W [H, H], b per further hidden layer, then Wo [H, nout], bo; the v block follows the pi block and log_std.
static void net_layout(const ml4ca_policy_cfg& cfg, int32_t net, GradArgs* a) {
  const int H = cfg.hidden, O = cfg.obs_dim, Ad = cfg.act_dim, NL = cfg.n_hidden;
  const int pi_size = O * H + H + (NL - 1) * (H * H + H) + H * Ad + Ad;
  a->obs = O, a->act = Ad, a->nout = net == 0 ? Ad : 1;
  a->hidden = H, a->n_hidden = NL;
  a->off_w[0] = net == 0 ? 0 : pi_size + Ad, a->off_b[0] = a->off_w[0] + O * H;
  for (int l = 1; l < NL; ++l) a->off_w[l] = a->off_b[l - 1] + H, a->off_b[l] = a->off_w[l] + H * H;
  a->off_w[NL] = a->off_b[NL - 1] + H, a->off_b[NL] = a->off_w[NL] + H * a->nout;
  a->off_ls = pi_size;
}

static int ppo_launch_fp32(const GradArgs& a, int activation, int net, cudaStream_t st) {
  const int64_t tiles = (a.n * (int64_t)a.T + ppo::TS - 1) / ppo::TS;
  const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
  const size_t smem = sizeof(ppo::Smem);
#define ML4CA_PPO_LAUNCH(ACTV, NETV)                                                                             \
  do {                                                                                                           \
    auto k = ppo::ppo_grad_kernel<ACTV, NETV>;                                                                   \
    ML4CA_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                 \
    k<<<grid, 256, smem, st>>>(a);                                                                               \
  } while (0)
  if (activation == 1) {
    if (net == 0) ML4CA_PPO_LAUNCH(1, 0); else ML4CA_PPO_LAUNCH(1, 1);
  } else {
    if (net == 0) ML4CA_PPO_LAUNCH(0, 0); else ML4CA_PPO_LAUNCH(0, 1);
  }
#undef ML4CA_PPO_LAUNCH
  return check_launch("ppo_grad_kernel");
}

// The pass behind ml4ca_ppo_grad_ex, ml4ca_trpo_policy_mu and ml4ca_trpo_kl_grad.  `a` arrives with the buffers, the loss mode and
// ctl / iter; tensor_cores is the process-wide switch that applies to the pass.  A gradient pass (grad != NULL) zeroes grad and
// stats, also when the batch is empty.  The tcgen05 kernel (fp16 operands, fp32 TMEM accumulation) runs when the switch is on;
// otherwise the fp32 CUDA-core kernels: ppo_grad_kernel for the 64 x 64 config, the generic one for the other shapes.
static int grad_pass(ml4ca_policy* p, int32_t net, int64_t n, int32_t T, GradArgs a, bool tensor_cores, cudaStream_t st) {
  ML4CA_REQUIRE(p != nullptr, "policy is NULL");
  ML4CA_REQUIRE(n >= 0 && T >= 0, "bad sizes");
  ml4ca_policy_cfg cfg;
  int32_t device = 0;
  int rc = ml4ca_policy_describe(p, &cfg, &device);
  if (rc != ML4CA_OK) return rc;
  if (a.grad != nullptr) {
    ML4CA_CUDA(cudaMemsetAsync(a.grad, 0, sizeof(float) * (size_t)ml4ca_policy_num_params(&cfg), st));
    ML4CA_CUDA(cudaMemsetAsync(a.stats, 0, sizeof(double) * 8, st));
  }
  if (n * (int64_t)T == 0) return ML4CA_OK;
  net_layout(cfg, net, &a);
  a.params = ml4ca_policy_params(p), a.n = n, a.T = T;
  if (tensor_cores && ml4ca_ppo_tc_supports(cfg.hidden, cfg.n_hidden, cfg.obs_dim, cfg.act_dim)) {
    __half* blob = nullptr;
    rc = tc_blob(device, &blob);
    if (rc != ML4CA_OK) return rc;
    return ml4ca_ppo_grad_tc_launch(a, cfg.activation, net, blob, st);
  }
  if (cfg.hidden == ppo::H && cfg.n_hidden == 2 && cfg.obs_dim <= ppo::XR) return ppo_launch_fp32(a, cfg.activation, net, st);
  return ml4ca_ppo_grad_generic_launch(a, cfg.activation, net, st);
}

extern "C" {

int ml4ca_ppo_grad(ml4ca_policy* p, int32_t net, int64_t n, int32_t T, const float* obs, const float* act, const float* adv,
                   const float* ret, const float* logp_old, float clip_ratio, float* grad, double* stats, void* stream) {
  return ml4ca_ppo_grad_ex(p, net, n, T, obs, act, adv, ret, logp_old, clip_ratio, grad, stats, nullptr, 0, stream);
}

int ml4ca_ppo_ctl_begin(ml4ca_ppo_ctl* ctl, void* stream) {
  ML4CA_REQUIRE(ctl != nullptr, "ctl is NULL");
  ppo::ppo_ctl_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(ctl, 1, 0, 0);
  return check_launch("ppo_ctl_kernel");
}

int ml4ca_ppo_ctl_end(ml4ca_ppo_ctl* ctl, int32_t pi_iters, int32_t v_iters, void* stream) {
  ML4CA_REQUIRE(ctl != nullptr && pi_iters >= 1 && v_iters >= 0, "bad arguments");
  ppo::ppo_ctl_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(ctl, 0, pi_iters, v_iters);
  return check_launch("ppo_ctl_kernel");
}

int ml4ca_adam_step_dev(int64_t m, float* params, const float* grad, float* m1, float* m2, float lr, float beta1, float beta2,
                        float eps, float grad_scale, int32_t net, int32_t iter, const float* stats_tail, float count,
                        float kl_limit, ml4ca_ppo_ctl* ctl, void* stream) {
  ML4CA_REQUIRE(m >= 0 && params && grad && m1 && m2 && stats_tail && ctl && iter >= 0 && (net == 0 || net == 1) && count > 0.f,
                "bad arguments");
  if (m == 0) return ML4CA_OK;
  ppo::adam_dev_kernel<<<(unsigned)((m + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      m, params, grad, m1, m2, lr, beta1, beta2, eps, grad_scale, net, iter, stats_tail, count, kl_limit, ctl);
  return check_launch("adam_dev_kernel");
}

int ml4ca_ppo_grad_ex(ml4ca_policy* p, int32_t net, int64_t n, int32_t T, const float* obs, const float* act, const float* adv,
                      const float* ret, const float* logp_old, float clip_ratio, float* grad, double* stats,
                      const ml4ca_ppo_ctl* ctl, int32_t iter, void* stream) {
  ML4CA_REQUIRE(p != nullptr && grad != nullptr && stats != nullptr && obs != nullptr, "policy, obs, grad and stats are required");
  ML4CA_REQUIRE(net == 0 || net == 1, "net: 0 = pi, 1 = v");
  if (net == 0) ML4CA_REQUIRE(act && adv && logp_old, "pi pass needs act, adv and logp_old");
  else ML4CA_REQUIRE(ret != nullptr, "v pass needs ret");
  GradArgs a = {};
  a.obs_buf = obs, a.act_buf = act, a.adv = adv, a.logp_old = logp_old, a.ret = ret;
  a.clip = clip_ratio;
  a.grad = grad, a.stats = stats;
  a.ctl = reinterpret_cast<const int32_t*>(ctl), a.iter = iter;
  return grad_pass(p, net, n, T, a, !g_use_fp32, static_cast<cudaStream_t>(stream));
}

int ml4ca_trpo_policy_mu(ml4ca_policy* p, int64_t n, int32_t T, const float* obs, float* mu, void* stream) {
  ML4CA_REQUIRE(obs != nullptr && mu != nullptr, "obs and mu are required");
  GradArgs a = {};
  a.obs_buf = obs, a.mu_out = mu;
  return grad_pass(p, 0, n, T, a, g_trpo_tc, static_cast<cudaStream_t>(stream));
}

int ml4ca_trpo_kl_grad(ml4ca_policy* p, int64_t n, int32_t T, const float* obs, const float* mu_old, const float* log_std_old,
                       float* grad, double* stats, void* stream) {
  ML4CA_REQUIRE(obs && mu_old && log_std_old && grad && stats, "obs, mu_old, log_std_old, grad and stats are required");
  GradArgs a = {};
  a.obs_buf = obs, a.act_buf = mu_old, a.kl_ls_old = log_std_old, a.loss_mode = 1;
  a.grad = grad, a.stats = stats;
  return grad_pass(p, 0, n, T, a, g_trpo_tc, static_cast<cudaStream_t>(stream));
}

int ml4ca_adam_step(int64_t m, float* params, const float* grad, float* m1, float* m2, float lr, float beta1, float beta2,
                    float eps, int32_t t, float grad_scale, void* stream) {
  ML4CA_REQUIRE(m >= 0 && params && grad && m1 && m2 && t >= 1, "bad arguments");
  if (m == 0) return ML4CA_OK;
  const double lr_t = (double)lr * sqrt(1.0 - pow((double)beta2, (double)t)) / (1.0 - pow((double)beta1, (double)t));
  ppo::adam_kernel<<<(unsigned)((m + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(m, params, grad, m1, m2, (float)lr_t,
                                                                                             beta1, beta2, eps, grad_scale);
  return check_launch("adam_kernel");
}

}  // extern "C"
