// ppo_update_generic.cu -- K6 for the reference's OWN network shapes: hidden 80 x 80 x 80 (train.py:30-32, every shipped
// checkpoint but one) and 64 x 64 x 64 (models/limited), next to the 64 x 64 of the BASELINE config that ppo_update.cu /
// ppo_update_tc.cu specialise.
//
// Same contract as ppo_grad_kernel (ppo_update.cu; reference ppo.py:234-250, core.py:29-46): forward, loss and backward
// of ONE network (NET 0 = pi incl. log_std, 1 = v) over every sample of a [T, ., n] buffer in fp32, gradient SUMS into the
// flat vector, loss statistics in double; also the TRPO passes (loss_mode 1 = d_kl, mu_out = forward only).
// Hidden 64 x 64, 64^3 and 80^3 (the networks ml4ca_policy_create accepts), obs <= 16.  A persistent CTA (8 warps) works on
// tiles of 64 samples; the three GEMM shapes of a layer are register-tiled so that a fused multiply-add costs 0.2 .. 0.4
// shared-memory loads (the first version of this kernel had no register tiling, 2 loads per FMA, and ran at the shared-memory
// bandwidth: 83 M sample-passes/s):
//   forward        h_l[j][s] = f(b_l[j] + sum_k h_{l-1}[k][s] W_l[k][j])     warp w owns HP/8 features, a lane two samples:
//                                                                            per k two activation loads + HP/16 64-bit weight loads
//   weight grad.   dW_l[k][j] += sum_s h_{l-1}[k][s] g_l[j][s]               thread (k-block, j-block) owns a (HP/16)^2 tile of
//                                                                            dW_l IN REGISTERS for the whole launch (16 x 16 tiles
//                                                                            = 256 threads); bias gradients ride on the first k-block
//   backward data  g_{l-1}[k][s] = f'(h_{l-1}[k][s]) sum_j W_l[k][j] g_l[j][s]   warp w owns HP/8 rows k, a lane two samples:
//                                                                            per 4 j: 8 signal loads + HP/8 128-bit weight loads
// HP = the width rounded up to 64 / 80 (template parameter: the register tiles need compile-time shapes).  The weights are
// copied to shared memory ZERO-PADDED to HP, so every row / column offset is an immediate and nothing on the path is masked.
// Weights, activations and back-propagated signals live in shared memory (80^3: 173 KB); activation rows have stride 66: a
// lane's two samples are one 64-bit access, conflict-free both for lane = sample reads and for the strided tiles of the
// weight-gradient step (neighbouring threads read neighbouring rows: banks 2 t, 2 t + 1).  The weight-gradient accumulators are
// flushed once per launch with atomicAdd.  Measured (B200, 80^3, 1.6 M samples): 83 -> 171 (register tiles) -> 314 (padded,
// immediate offsets) -> see profiles/ppo_grad_r2.md for the shipped figure.
//
// This kernel is fp32 on the CUDA cores: coverage of the reference's shapes with 1e-4 gradients.  The throughput path for
// millions of samples stays the tcgen05 kernel of the 64 x 64 config.
#include <stdlib.h>

#include "common.h"
#include "ppo_grad.h"

namespace ml4ca {
namespace generic {

constexpr int TS = 64;     // samples per tile: lane s owns samples 2 s and 2 s + 1 (one 64-bit access)
constexpr int RS = 66;     // activation row stride (floats): even, so sample pairs are 8-byte aligned in every row
constexpr int OP = 8;      // padded output width (act_dim <= 7, value head 1)
constexpr int NW = 8;      // warps per CTA
constexpr int NT = NW * 32;

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

__host__ __device__ inline int padded_width(int H) { return H <= 64 ? 64 : 80; }

// The net's parameters in shared memory, ZERO-PADDED to the compile-time width HP: W1 [obs][HP], b1 [HP], then per further hidden
// layer W_l [HP][HP], b_l [HP], then Wo [HP][OP], bo [OP].  Every row / column offset is a compile-time constant (immediate
// operands instead of index arithmetic with a run-time H), and padded features need no masks anywhere: their weights and biases
// are zero, so their activations and back-propagated signals are zero.
__host__ __device__ inline int padded_params(int obs, int HP, int NL) { return (obs + 1) * HP + (NL - 1) * (HP * HP + HP) + HP * OP + OP; }

// shared-memory plan (floats): padded parameters, dOUT transposed [TS x OP] (128-bit reads), activations of layers 0..NL
// [(obs + NL HP) x RS], two back-propagated signals [2 x HP x RS], out / dOUT [OP x RS], actions [OP x RS], aux [2 x RS],
// per-output constants [5 x OP].
__host__ __device__ inline size_t smem_floats(int obs, int H, int NL) {
  const int HP = padded_width(H);
  return (size_t)padded_params(obs, HP, NL) + (size_t)TS * OP + (size_t)(obs + NL * HP) * RS + (size_t)2 * HP * RS + (size_t)2 * OP * RS +
         2 * RS + 5 * OP + 8;
}

// Feature (forward) / row (backward data) jj of warp w: eight consecutive ones from the first 64, the rest from the tail, so
// that a warp's slice of a weight row is two 128-bit words plus one 64-bit word (HP = 80).
template <int JT>
__device__ __forceinline__ int warp_feature(int w, int jj) { return jj < 8 ? w * 8 + jj : 64 + (JT - 8) * w + (jj - 8); }
template <int JT>
__device__ __forceinline__ void load_slice(const float* __restrict__ row, int w, float (&v)[JT]) {
  const float4 a = *reinterpret_cast<const float4*>(row + w * 8), b = *reinterpret_cast<const float4*>(row + w * 8 + 4);
  v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y, v[6] = b.z, v[7] = b.w;
  if constexpr (JT == 10) {
    const float2 c = *reinterpret_cast<const float2*>(row + 64 + 2 * w);
    v[8] = c.x, v[9] = c.y;
  }
}

template <int ACTIVATION, int NET, int HP>
__global__ void __launch_bounds__(NT, 1) ppo_grad_generic_kernel(const GradArgs A) {
  if (A.ctl != nullptr && A.ctl[0] != 0 && A.ctl[1] < A.iter) return;   // the policy loop has stopped (ml4ca_ppo_ctl)
  constexpr int JT = HP / 8;     // features (forward) / rows (backward data) per warp
  constexpr int BT = HP / 16;    // edge of a thread's weight-gradient tile
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int obs = A.obs, H = A.hidden, NL = A.n_hidden, nout = A.nout;
  float* W = sm;                         // this net's parameters, zero-padded to HP (padded_params)
  const int PW = padded_params(obs, HP, NL);
  float* doutT = W + PW;                 // dOUT [s][OP]
  float* act0 = doutT + TS * OP;         // layer 0 = observation rows
  float* gbuf = act0 + (size_t)(obs + NL * HP) * RS;
  float* out = gbuf + (size_t)2 * HP * RS;
  float* actb = out + OP * RS;
  float* aux = actb + OP * RS;           // adv | ret, logp_old
  float* cst = aux + 2 * RS;             // sd, inv, ls, kiv, kls [OP each]
  auto layer_in = [&](int l) { return l == 0 ? obs : H; };                    // fan-in of layer l (0-based; l == NL: output)
  auto w_off = [&](int l) {                                                    // offset of W_l inside the net's block
    int o = 0;
    for (int q = 0; q < l; ++q) o += layer_in(q) * H + H;
    return o;
  };
  auto wp_off = [&](int l) { return l == 0 ? 0 : (obs + 1) * HP + (l - 1) * (HP * HP + HP); };   // the same in the padded copy
  auto act_rows = [&](int l) { return act0 + (size_t)(l == 0 ? 0 : obs + (l - 1) * HP) * RS; };  // activations entering layer l

  for (int e = tid; e < (int)smem_floats(obs, H, NL); e += NT) sm[e] = 0.f;
  __syncthreads();
  for (int l = 0; l <= NL; ++l) {          // flat order W1 [obs,H], b1, W2 [H,H], b2, ..., Wo [H,nout], bo -> padded rows
    const int K = layer_in(l), N = (l == NL) ? nout : H, NP = (l == NL) ? OP : HP;
    const float* src = A.params + A.off_w[0] + w_off(l);
    float* dst = W + wp_off(l);
    for (int e = tid; e < (K + 1) * N; e += NT) {
      const int k = e / N, j = e - k * N;
      dst[(k < K ? k * NP : (l == 0 ? obs : HP) * NP) + j] = src[e];       // row K of the flat block is the bias
    }
  }
  if (tid < OP) {
    const float ls = (NET == 0 && tid < nout) ? A.params[A.off_ls + tid] : 0.f;
    const float sd = expf(ls);
    cst[tid] = sd, cst[OP + tid] = 1.0f / (sd + 1e-8f), cst[2 * OP + tid] = ls;
    const float lo = (NET == 0 && A.loss_mode == 1 && tid < nout) ? A.kl_ls_old[tid] : 0.f;
    cst[3 * OP + tid] = 1.0f / (expf(2.0f * lo) + 1e-8f), cst[4 * OP + tid] = lo;                 // trpo/core.py:57-58
  }
  // weight-gradient accumulators (registers, whole launch): thread (kb, jb) owns rows kb*BT.., columns jb*BT.. of every
  // hidden-to-hidden dW, row kb (< obs) of dW1, and -- kb == 0 -- the bias gradients of its columns; thread t < H owns row t of dWo
  const int kb = tid >> 4, jb = tid & 15;
  float accH[2][BT * BT], acc1[BT], accB[3][BT], accO[OP], accBo = 0.f;
#pragma unroll
  for (int q = 0; q < 2; ++q)
#pragma unroll
    for (int e = 0; e < BT * BT; ++e) accH[q][e] = 0.f;
#pragma unroll
  for (int e = 0; e < BT; ++e) acc1[e] = 0.f, accB[0][e] = 0.f, accB[1][e] = 0.f, accB[2][e] = 0.f;
#pragma unroll
  for (int o = 0; o < OP; ++o) accO[o] = 0.f;
  float dls_a[OP];                       // warps 0-1, lane = sample: sum over its samples of dL/dlog_std[a]
#pragma unroll
  for (int o = 0; o < OP; ++o) dls_a[o] = 0.f;
  double st[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  __syncthreads();

  const int64_t n = A.n;
  const int64_t total = n * (int64_t)A.T;       // tiles run over the flat sample index (common.h: split_sample)
  const int64_t num_tiles = (total + TS - 1) / TS;
  // The rows of a tile (observation, action / return, advantage, old log-likelihood) are fetched ONE TILE AHEAD into registers
  // (warp w: rows w, w + 8, ...; a lane two samples, coalesced) and written to shared memory when the previous tile has
  // finished with them: their HBM latency is off the tile's chain.
  const int rows_in = obs + (NET == 0 ? A.act + 2 : 1);
  constexpr int RPW = 4;                        // rows per warp: obs <= 16, act <= 8, + 2
  int64_t tN[2] = {0, 0}, iN[2] = {0, 0};
  bool liveN[2] = {false, false};
  float pre[RPW][2];
  auto row_slot = [&](int row, float*& dst) {   // where row `row` of a tile lives in shared memory
    if (row < obs) dst = act0 + (size_t)row * RS;
    else if (NET == 1) dst = aux;
    else if (row < obs + A.act) dst = actb + (size_t)(row - obs) * RS;
    else if (row == obs + A.act) dst = aux;
    else dst = aux + RS;
  };
  auto prefetch = [&](int64_t tile) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int64_t smp = tile * TS + q * 32 + lane;
      liveN[q] = smp < total;
      tN[q] = 0, iN[q] = 0;
      if (liveN[q]) split_sample(smp, n, tN[q], iN[q]);
    }
#pragma unroll
    for (int r = 0; r < RPW; ++r) {
      const int row = warp + NW * r;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int64_t t = tN[q], i = iN[q];
        const float* base = nullptr;
        int64_t off = 0;
        if (row < obs) base = A.obs_buf, off = ((int64_t)t * obs + row) * n;
        else if (row >= rows_in) base = nullptr;
        else if (NET == 1) base = A.ret, off = (int64_t)t * n;
        else if (row < obs + A.act) base = A.act_buf, off = ((int64_t)t * A.act + (row - obs)) * n;
        else if (row == obs + A.act) base = A.adv, off = (int64_t)t * n;
        else base = A.logp_old, off = (int64_t)t * n;
        pre[r][q] = (base != nullptr && liveN[q]) ? __ldg(base + off + i) : 0.f;
      }
    }
  };
  if ((int64_t)blockIdx.x < num_tiles) prefetch(blockIdx.x);
  for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    int64_t t2[2], i2[2];
    bool live2[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) t2[q] = tN[q], i2[q] = iN[q], live2[q] = liveN[q];
#pragma unroll
    for (int r = 0; r < RPW; ++r) {
      const int row = warp + NW * r;
      if (row < rows_in) {
        float* dst;
        row_slot(row, dst);
        dst[lane] = pre[r][0], dst[32 + lane] = pre[r][1];
      }
    }
    __syncthreads();
    if (tile + gridDim.x < num_tiles) prefetch(tile + gridDim.x);
    // ---- forward -----------------------------------------------------------------------------------------------------------
#pragma unroll 1
    for (int l = 0; l < NL; ++l) {
      const int K = layer_in(l);
      const float* in = act_rows(l);
      float* o = act_rows(l + 1);
      const float* wr = W + wp_off(l);               // row k of W_l at wr + k * HP, the bias row behind the K weight rows
      float a0[JT], a1[JT];
      load_slice<JT>(wr + (size_t)(l == 0 ? obs : HP) * HP, warp, a0);
#pragma unroll
      for (int jj = 0; jj < JT; ++jj) a1[jj] = a0[jj];
#pragma unroll 4
      for (int k = 0; k < K; ++k) {
        const float2 x = *reinterpret_cast<const float2*>(in + (size_t)k * RS + 2 * lane);
        float w[JT];
        load_slice<JT>(wr + k * HP, warp, w);
#pragma unroll
        for (int jj = 0; jj < JT; ++jj) a0[jj] = fmaf(x.x, w[jj], a0[jj]), a1[jj] = fmaf(x.y, w[jj], a1[jj]);
      }
#pragma unroll
      for (int jj = 0; jj < JT; ++jj)
        *reinterpret_cast<float2*>(o + (size_t)warp_feature<JT>(warp, jj) * RS + 2 * lane) =
            make_float2(act_fn<ACTIVATION>(a0[jj]), act_fn<ACTIVATION>(a1[jj]));
      __syncthreads();
    }
    {
      const float* in = act_rows(NL);
      const float* Wo = W + wp_off(NL);
      const float* bo = Wo + HP * OP;
      for (int j = warp; j < nout; j += NW) {
        float c0 = bo[j], c1 = c0;
#pragma unroll 8
        for (int k = 0; k < HP; ++k) {
          const float w = Wo[k * OP + j];
          const float2 x = *reinterpret_cast<const float2*>(in + (size_t)k * RS + 2 * lane);
          c0 = fmaf(x.x, w, c0), c1 = fmaf(x.y, w, c1);
        }
        *reinterpret_cast<float2*>(out + (size_t)j * RS + 2 * lane) = make_float2(c0, c1);
      }
    }
    __syncthreads();
    if (A.mu_out != nullptr) {           // forward only (uniform branch): store the means, next tile
      for (int a = warp; a < nout; a += NW)
#pragma unroll
        for (int q = 0; q < 2; ++q)
          if (live2[q]) A.mu_out[((int64_t)t2[q] * nout + a) * n + i2[q]] = out[(size_t)a * RS + q * 32 + lane];
      __syncthreads();
      continue;
    }
    // ---- loss and dOUT (sum convention), warps 0-1: thread = sample -----------------------------------------------------------
    if (warp < 2) {
      const int s = tid;
      const bool live = live2[warp];
      const float *sd = cst, *inv = cst + OP, *ls = cst + 2 * OP, *kiv = cst + 3 * OP, *kls = cst + 4 * OP;
      float dout[OP];
#pragma unroll
      for (int a = 0; a < OP; ++a) dout[a] = 0.f;
      if (NET == 0 && A.loss_mode == 1) {
        // d_kl = mean_s sum_a 0.5 (((mu_old - mu)^2 + var) / (var_old + EPS) - 1) + log_std_old - log_std   (trpo/core.py:52-60)
        double kl = 0.0;
#pragma unroll
        for (int a = 0; a < OP; ++a) {
          if (a < nout) {
            const float d = out[(size_t)a * RS + s] - actb[(size_t)a * RS + s], var = sd[a] * sd[a];
            kl += (double)(0.5f * ((d * d + var) * kiv[a] - 1.0f) + (kls[a] - ls[a]));
            dout[a] = live ? d * kiv[a] : 0.f;
            dls_a[a] += live ? (var * kiv[a] - 1.0f) : 0.f;
          }
        }
        if (live) st[2] += kl;
      } else if constexpr (NET == 0) {
        float logp = 0.f, z[OP];
#pragma unroll
        for (int a = 0; a < OP; ++a) {
          z[a] = 0.f;
          if (a < nout) {
            z[a] = (actb[(size_t)a * RS + s] - out[(size_t)a * RS + s]) * inv[a];     // (x - mu) / (exp(log_std) + EPS), core.py:45
            logp += -0.5f * (z[a] * z[a] + 2.0f * ls[a] + 1.8378770664093453f);
          }
        }
        const float adv = aux[s], lpo = aux[RS + s];
        const float ratio = expf(logp - lpo);                                        // ppo.py:234
        const float min_adv = adv > 0.f ? (1.0f + A.clip) * adv : (1.0f - A.clip) * adv;   // :235
        const float ra = ratio * adv;
        const bool use_ratio = ra <= min_adv;                                        // tf.minimum sends the gradient to x where x <= y
        const float dlogp = (live && use_ratio) ? -ra : 0.f;
#pragma unroll
        for (int a = 0; a < OP; ++a) {
          if (a < nout) {
            dout[a] = dlogp * z[a] * inv[a];                                          // dlogp/dmu = (x - mu) / (std + EPS)^2
            dls_a[a] += dlogp * (z[a] * z[a] * sd[a] * inv[a] - 1.0f);                // dlogp/dlog_std = z^2 std / (std + EPS) - 1
          }
        }
        if (live) {
          st[0] += (double)fminf(ra, min_adv);
          const float dl = lpo - logp;
          st[2] += 0.5 * (double)dl * (double)dl;                                    // :242
          st[3] += (double)(-logp);                                                  // :243
          st[4] += (ratio > 1.0f + A.clip || ratio < 1.0f - A.clip) ? 1.0 : 0.0;     // :244
        }
      } else {
        const float v = out[s], r = aux[s];
        const float e = v - r;
        dout[0] = live ? 2.0f * e : 0.f;                                             // d(ret - v)^2 / dv
        if (live) st[1] += (double)e * (double)e;                                    // :236
      }
#pragma unroll
      for (int a = 0; a < OP; ++a) out[(size_t)a * RS + s] = dout[a];
      *reinterpret_cast<float4*>(doutT + s * OP) = make_float4(dout[0], dout[1], dout[2], dout[3]);
      *reinterpret_cast<float4*>(doutT + s * OP + 4) = make_float4(dout[4], dout[5], dout[6], dout[7]);
    }
    __syncthreads();
    // ---- backward ------------------------------------------------------------------------------------------------------------
    // output layer: dWo, dbo, g_NL = (dOUT Wo^T) .* f'(h_NL)
    float* g_cur = gbuf;
    float* g_nxt = gbuf + (size_t)HP * RS;
    {
      const float* hin = act_rows(NL);
      const float* Wo = W + wp_off(NL);
      if (tid < H) {
        const float* hp = hin + (size_t)tid * RS;
#pragma unroll 2
        for (int s = 0; s < TS; s += 2) {
          const float2 hv = *reinterpret_cast<const float2*>(hp + s);
          const float4 d0 = *reinterpret_cast<const float4*>(doutT + s * OP), d1 = *reinterpret_cast<const float4*>(doutT + s * OP + 4);
          const float4 e0 = *reinterpret_cast<const float4*>(doutT + s * OP + 8), e1 = *reinterpret_cast<const float4*>(doutT + s * OP + 12);
          accO[0] = fmaf(hv.x, d0.x, accO[0]), accO[1] = fmaf(hv.x, d0.y, accO[1]), accO[2] = fmaf(hv.x, d0.z, accO[2]);
          accO[3] = fmaf(hv.x, d0.w, accO[3]), accO[4] = fmaf(hv.x, d1.x, accO[4]), accO[5] = fmaf(hv.x, d1.y, accO[5]);
          accO[6] = fmaf(hv.x, d1.z, accO[6]), accO[7] = fmaf(hv.x, d1.w, accO[7]);
          accO[0] = fmaf(hv.y, e0.x, accO[0]), accO[1] = fmaf(hv.y, e0.y, accO[1]), accO[2] = fmaf(hv.y, e0.z, accO[2]);
          accO[3] = fmaf(hv.y, e0.w, accO[3]), accO[4] = fmaf(hv.y, e1.x, accO[4]), accO[5] = fmaf(hv.y, e1.y, accO[5]);
          accO[6] = fmaf(hv.y, e1.z, accO[6]), accO[7] = fmaf(hv.y, e1.w, accO[7]);
        }
      } else if (tid >= HP && tid < HP + nout) {
        const float* dp = out + (size_t)(tid - HP) * RS;
        float acc = 0.f;
        for (int s = 0; s < TS; ++s) acc += dp[s];
        accBo += acc;
      }
      float d0[OP], d1[OP];
      {
        const float4 u0 = *reinterpret_cast<const float4*>(doutT + 2 * lane * OP), u1 = *reinterpret_cast<const float4*>(doutT + 2 * lane * OP + 4);
        const float4 v0 = *reinterpret_cast<const float4*>(doutT + (2 * lane + 1) * OP), v1 = *reinterpret_cast<const float4*>(doutT + (2 * lane + 1) * OP + 4);
        d0[0] = u0.x, d0[1] = u0.y, d0[2] = u0.z, d0[3] = u0.w, d0[4] = u1.x, d0[5] = u1.y, d0[6] = u1.z, d0[7] = u1.w;
        d1[0] = v0.x, d1[1] = v0.y, d1[2] = v0.z, d1[3] = v0.w, d1[4] = v1.x, d1[5] = v1.y, d1[6] = v1.z, d1[7] = v1.w;
      }
#pragma unroll
      for (int kk = 0; kk < JT; ++kk) {
        const int k = warp_feature<JT>(warp, kk);
        const float4 wa = *reinterpret_cast<const float4*>(Wo + k * OP), wb = *reinterpret_cast<const float4*>(Wo + k * OP + 4);
        const float w[OP] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};      // padded outputs: zero weights, zero dOUT
        float c0 = 0.f, c1 = 0.f;
#pragma unroll
        for (int j = 0; j < OP; ++j) c0 = fmaf(w[j], d0[j], c0), c1 = fmaf(w[j], d1[j], c1);
        const float2 hv = *reinterpret_cast<const float2*>(hin + (size_t)k * RS + 2 * lane);
        *reinterpret_cast<float2*>(g_cur + (size_t)k * RS + 2 * lane) = make_float2(c0 * act_grad<ACTIVATION>(hv.x), c1 * act_grad<ACTIVATION>(hv.y));
      }
    }
    __syncthreads();
#pragma unroll
    for (int lu = 2; lu >= 0; --lu) {          // unrolled over the layer slot: the accumulators are indexed at compile time
      const int l = lu;
      if (l < NL) {
        const int K = layer_in(l);
        const float* hin = act_rows(l);
        const float* Wl = W + wp_off(l);
        // -- weight gradient of layer l
        // (strided tiles: rows kb + 16 kk, columns jb + 16 jj -- neighbouring threads read neighbouring rows: conflict-free)
        const float* gp = g_cur + (size_t)jb * RS;
        if (l > 0) {
          const float* hp = hin + (size_t)kb * RS;
#pragma unroll 2
          for (int s = 0; s < TS; s += 2) {
            float2 hv[BT], gv[BT];
#pragma unroll
            for (int e = 0; e < BT; ++e) {
              hv[e] = *reinterpret_cast<const float2*>(hp + (size_t)(16 * e) * RS + s);
              gv[e] = *reinterpret_cast<const float2*>(gp + (size_t)(16 * e) * RS + s);
            }
#pragma unroll
            for (int kk = 0; kk < BT; ++kk)
#pragma unroll
              for (int jj = 0; jj < BT; ++jj) {
                float& acc = accH[lu > 0 ? lu - 1 : 0][kk * BT + jj];
                acc = fmaf(hv[kk].x, gv[jj].x, acc), acc = fmaf(hv[kk].y, gv[jj].y, acc);
              }
            if (kb == 0) {
#pragma unroll
              for (int jj = 0; jj < BT; ++jj) accB[lu][jj] += gv[jj].x + gv[jj].y;
            }
          }
        } else if (kb < obs) {
          const float* hp = hin + (size_t)kb * RS;
#pragma unroll 2
          for (int s = 0; s < TS; s += 2) {
            const float2 hv = *reinterpret_cast<const float2*>(hp + s);
            float2 gv[BT];
#pragma unroll
            for (int e = 0; e < BT; ++e) gv[e] = *reinterpret_cast<const float2*>(gp + (size_t)(16 * e) * RS + s);
#pragma unroll
            for (int jj = 0; jj < BT; ++jj) acc1[jj] = fmaf(hv.x, gv[jj].x, acc1[jj]), acc1[jj] = fmaf(hv.y, gv[jj].y, acc1[jj]);
            if (kb == 0) {
#pragma unroll
              for (int jj = 0; jj < BT; ++jj) accB[0][jj] += gv[jj].x + gv[jj].y;
            }
          }
        }
        // -- back-propagated signal entering layer l - 1
        if (l > 0) {
          float c0[JT], c1[JT];
#pragma unroll
          for (int kk = 0; kk < JT; ++kk) c0[kk] = c1[kk] = 0.f;
#pragma unroll 2
          for (int j = 0; j < HP; j += 4) {
            float p0[4], p1[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float2 pv = *reinterpret_cast<const float2*>(g_cur + (size_t)(j + c) * RS + 2 * lane);
              p0[c] = pv.x, p1[c] = pv.y;
            }
#pragma unroll
            for (int kk = 0; kk < JT; ++kk) {
              const float4 w = *reinterpret_cast<const float4*>(Wl + warp_feature<JT>(warp, kk) * HP + j);
              c0[kk] = fmaf(w.x, p0[0], c0[kk]), c0[kk] = fmaf(w.y, p0[1], c0[kk]), c0[kk] = fmaf(w.z, p0[2], c0[kk]), c0[kk] = fmaf(w.w, p0[3], c0[kk]);
              c1[kk] = fmaf(w.x, p1[0], c1[kk]), c1[kk] = fmaf(w.y, p1[1], c1[kk]), c1[kk] = fmaf(w.z, p1[2], c1[kk]), c1[kk] = fmaf(w.w, p1[3], c1[kk]);
            }
          }
#pragma unroll
          for (int kk = 0; kk < JT; ++kk) {
            const int k = warp_feature<JT>(warp, kk);
            const float2 hv = *reinterpret_cast<const float2*>(hin + (size_t)k * RS + 2 * lane);
            *reinterpret_cast<float2*>(g_nxt + (size_t)k * RS + 2 * lane) = make_float2(c0[kk] * act_grad<ACTIVATION>(hv.x), c1[kk] * act_grad<ACTIVATION>(hv.y));
          }
        }
        __syncthreads();
        float* tmp = g_cur;
        g_cur = g_nxt, g_nxt = tmp;
      }
    }
  }

  if (A.mu_out != nullptr) return;       // forward-only pass (uniform)
  // ---- flush ---------------------------------------------------------------------------------------------------------------------
  float* grad = A.grad + A.off_w[0];
  {
    // layer 0: row kb of dW1, bias b1
#pragma unroll
    for (int jj = 0; jj < BT; ++jj) {
      const int j = jb + 16 * jj;
      if (j < H) {
        if (kb < obs && acc1[jj] != 0.f) atomicAdd(grad + kb * H + j, acc1[jj]);
        if (kb == 0 && accB[0][jj] != 0.f) atomicAdd(grad + obs * H + j, accB[0][jj]);
      }
    }
#pragma unroll
    for (int lu = 1; lu < 3; ++lu) {
      if (lu < NL) {
        const int off = w_off(lu);
#pragma unroll
        for (int kk = 0; kk < BT; ++kk)
#pragma unroll
          for (int jj = 0; jj < BT; ++jj) {
            const int k = kb + 16 * kk, j = jb + 16 * jj;
            const float v = accH[lu - 1][kk * BT + jj];
            if (k < H && j < H && v != 0.f) atomicAdd(grad + off + k * H + j, v);
          }
        if (kb == 0) {
#pragma unroll
          for (int jj = 0; jj < BT; ++jj) {
            const int j = jb + 16 * jj;
            if (j < H && accB[lu][jj] != 0.f) atomicAdd(grad + off + H * H + j, accB[lu][jj]);
          }
        }
      }
    }
    const int offo = w_off(NL);
    if (tid < H) {
#pragma unroll
      for (int j = 0; j < OP; ++j)
        if (j < nout && accO[j] != 0.f) atomicAdd(grad + offo + tid * nout + j, accO[j]);
    } else if (tid >= HP && tid < HP + nout) {
      if (accBo != 0.f) atomicAdd(grad + offo + H * nout + (tid - HP), accBo);
    }
  }
  if (warp < 2) {
#pragma unroll
    for (int a = 0; a < OP; ++a) {
      float r = dls_a[a];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, off);
      if (NET == 0 && lane == 0 && a < nout) atomicAdd(A.grad + A.off_ls + a, r);
    }
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      double r = st[q];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, off);
      if (lane == 0 && r != 0.0) atomicAdd(A.stats + q, r);
    }
    if (tid == 0 && blockIdx.x == 0) atomicAdd(A.stats + 5, (double)A.n * (double)A.T);
  }
}

}  // namespace generic
}  // namespace ml4ca

using namespace ml4ca;

template <int HP>
static int launch_generic(const GradArgs& a, int activation, int net, int grid, size_t smem, cudaStream_t st) {
#define ML4CA_PPOGEN_LAUNCH(ACTV, NETV)                                                                          \
  do {                                                                                                           \
    auto k = generic::ppo_grad_generic_kernel<ACTV, NETV, HP>;                                                   \
    ML4CA_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                 \
    k<<<grid, generic::NT, smem, st>>>(a);                                                                       \
  } while (0)
  if (activation == 1) {
    if (net == 0) ML4CA_PPOGEN_LAUNCH(1, 0); else ML4CA_PPOGEN_LAUNCH(1, 1);
  } else {
    if (net == 0) ML4CA_PPOGEN_LAUNCH(0, 0); else ML4CA_PPOGEN_LAUNCH(0, 1);
  }
#undef ML4CA_PPOGEN_LAUNCH
  return check_launch("ppo_grad_generic_kernel");
}

int ml4ca_ppo_grad_generic_launch(const GradArgs& a, int activation, int net, cudaStream_t st) {
  const bool shape = (a.hidden == 64 && (a.n_hidden == 2 || a.n_hidden == 3)) || (a.hidden == 80 && a.n_hidden == 3);
  ML4CA_REQUIRE(shape && a.obs >= 1 && a.obs <= 16 && a.nout <= generic::OP,
                "generic gradient kernel: hidden 64 x 64, 64^3 or 80^3, obs_dim <= 16, outputs <= 8");
  const int64_t tiles = (a.n * (int64_t)a.T + generic::TS - 1) / generic::TS;
  const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
  const size_t smem = sizeof(float) * generic::smem_floats(a.obs, a.hidden, a.n_hidden);
  ML4CA_REQUIRE(smem <= 227 * 1024, "network too large for the shared-memory plan of the generic gradient kernel");
  if (a.hidden == 64) return launch_generic<64>(a, activation, net, grid, smem, st);
  return launch_generic<80>(a, activation, net, grid, smem, st);
}
