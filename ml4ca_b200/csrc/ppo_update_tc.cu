// ppo_update_tc.cu -- K6 on the tensor cores: PPO policy / value gradients with tcgen05 MMAs and TMEM accumulators.
//
// Same contract as ppo_grad_kernel (ppo_update.cu; reference ppo.py:234-250, core.py:29-46): forward, loss and
// backward of ONE network over every sample of a [T, ., n] buffer, gradient SUMS into the flat vector.  Shapes (template
// parameters H, NL): 64 x 64 (the BASELINE config), and the reference's own 80 x 80 x 80 (train.py:30-32) and 64 x 64 x 64.
// The text below spells out the 64 x 64 case; a deeper net repeats the hidden stage (one more forward GEMM, one more
// weight-gradient accumulator, one more backward-data GEMM per layer), a wider one has KP = H + 16 = 96 operand columns.
// All GEMMs of a 128-sample tile (seven for two hidden layers, ten for three) run as tcgen05.mma (fp16 operands in shared
// memory, fp32 accumulation in tensor memory); the CUDA cores only do the activation / loss epilogues:
//
//   forward      D = A0 B1^T          [128 x 16] x [64 x 16]^T      A0 = obs, 1 (bias column), pad
//                D = A1 B2^T          [128 x 80] x [64 x 80]^T      A1 = f(D), 1, pad
//                D = A2 Bo^T          [128 x 80] x [16 x 80]^T      -> mu / v
//   loss         per-sample dOUT (fp32), scaled by 64 and rounded to fp16 -> G3 [128 x 16]
//   backward     dWo  += A2^T G3      M = features, N = 16, K = 128 samples     (persistent TMEM accumulator)
//                D     = G3 WoT^T     -> G2 = D .* f'(H2)
//                dW2  += A1^T G2      M = features, N = 64, K = samples          (persistent)
//                D     = G2 W2n^T     -> G1 = D .* f'(H1)
//                dW1T += G1^T A0      M = hidden units, N = 16, K = samples      (persistent)
//
// The weight-gradient GEMMs reduce over the SAMPLE dimension.  Their operands are the very buffers the forward /
// backward-data GEMMs use, read through MN-major descriptors: in the canonical no-swizzle layout element (row r,
// column c) lives at (r/8) SBO + (c/8) 128 B + (r%8) 16 B + (c%8) 2 B, which is at the same time a K-major tile
// over (rows, columns) and an MN-major tile over (columns, rows) with the two strides exchanged -- no transposed
// copies are written.  With M fixed at 128 the transposed views read past the real feature count into neighbouring
// rows of the same buffer; those accumulator rows are garbage and are never flushed (rows are independent).
//
// Bias gradients fall out of the constant-1 columns (row H of dWo / dW2, column obs of dW1T).  Weight-gradient
// accumulators stay in TMEM for all tiles of the CTA (persistent grid) and are flushed once.  Tile groups of 128 threads
// (thread = sample = TMEM lane) run out of phase; an elected lane of the first two warps of a group issues its MMA chains
// (independent chains of a stage go to different issuers: one thread's MMAs run strictly one after the other).  Groups per
// CTA: three for 64 x 64, two for 64^3; 80^3 has two variants picked by the batch size (struct Shape below): two groups that
// share one set of weight-gradient accumulators (large batches: 5.1 G sample-passes/s), or one group with two threads per
// sample row (up to two waves of tiles: the shorter launch).  Measurements and dead ends: profiles/ppo_grad_r2.md.
//
// Numerics: fp16 operands (activations, weights, back-propagated signals x 64), fp32 accumulation: gradients agree
// with the float64 oracle to ~1e-3 of the largest component for two hidden layers, 4.5e-3 stated for three (the rounding
// enters once per layer; tests/test_ppo_update_gpu.py); the fp32 CUDA-core kernels (ppo_update.cu for 64 x 64 with obs_dim
// <= 12, ppo_update_generic.cu for the other networks) remain available (ML4CA_PPO_FP32=1) where 1e-4 .. 1e-5 is wanted.
#include <stdlib.h>

#include <cuda_fp16.h>

#include "common.h"
#include "ppo_grad.h"
#include "tc05.cuh"

namespace ml4ca {
namespace ppotc {

using namespace tc05;

constexpr int TS = 128, OP = 16;
constexpr float kScale = 64.0f;            // loss scaling of the back-propagated signals (fp16 range)

// Sizes, shared-memory plan and tensor-memory plan of one network shape (H hidden units, NL hidden layers).
// SH: the variant with tile groups on SHARED weight-gradient accumulators (80^3, large batches); false: every group owns its
// accumulators
template <int H_, int NL_, bool SH_ = false>
struct Shape {
  static constexpr int H = H_, NL = NL_, KP = H_ + 16;
  // tile groups per CTA: 3 x 64 KB (64 x 64), 2 x 84 KB (64^3), 1 x 100 KB or -- SHARED -- 2 x 80 KB (80^3)
#ifndef ML4CA_TC_G64X2
#define ML4CA_TC_G64X2 3     // tuning knobs (tools/kernel_variants.sh): groups / threads per row of the 64 x 64 and 64^3 shapes
#endif
#ifndef ML4CA_TC_SPLIT64X2
#define ML4CA_TC_SPLIT64X2 1
#endif
#ifndef ML4CA_TC_SPLIT64X3
#define ML4CA_TC_SPLIT64X3 1
#endif
  // SHARED (80^3): two groups do not fit side by side -- 2 x 100 KB of operand buffers, 2 x 272 TMEM columns.  They fit when
  //  * the back-propagated signal G_l is written IN PLACE over the activations A_l it is computed from (same thread, same
  //    addresses, layout of A_l: no G buffer), and
  //  * both groups accumulate into ONE set of weight-gradient accumulators (TMEM: 2 x 80 + 192 columns).  MMAs into the same
  //    accumulator must not be in flight from two issuing threads at once: a weight-gradient chain is issued under a CTA-wide
  //    lock (shared-memory word) that its group releases when the chain has completed (the wait every stage ends with).
  static constexpr bool SHARED = SH_ && H_ == 80 && NL_ == 3;
  static constexpr int G = (H_ == 64 && NL_ == 2) ? ML4CA_TC_G64X2 : ((H_ == 80 && NL_ == 3) ? (SHARED ? 2 : 1) : 2);
  // threads per sample row: with a single group nothing overlaps its epilogues, so two threads share a row (two warps may read
  // the same TMEM lane quadrant: warp w reaches lanes 32 (w % 4) ..) and each converts half of the accumulator columns
  static constexpr int SPLIT = (G == 1) ? 2 : ((H_ == 64 && NL_ == 2) ? ML4CA_TC_SPLIT64X2 : ML4CA_TC_SPLIT64X3);
  static constexpr int C_SPLIT = (H_ == 80) ? 48 : H_ / 2;     // columns [0, C_SPLIT) to the first thread of a row (multiple of 16)
  static constexpr int GT = 128 * SPLIT;                        // threads of a group
  static constexpr int THREADS = G * GT;
  // ---- shared memory: per group A0 | A_1 .. A_NL (activations entering layers 2 .. NL and the output layer) | G_out | G_hidden
  static constexpr int A0_B = TS * 16 * 2, AH_B = TS * KP * 2, GO_B = TS * 16 * 2, GH_B = TS * H * 2;
  static constexpr int GROUP_B = A0_B + NL * AH_B + GO_B + (SHARED ? 0 : GH_B);
  // operand images: B1 | B_2 .. B_NL | Bo | WoT | Wn_2 .. Wn_NL
  static constexpr int B1_E = H * 16, BH_E = H * KP, BO_E = OP * KP, WOT_E = H * 16, WN_E = H * H;
  static constexpr int BLOB_E = B1_E + (NL - 1) * BH_E + BO_E + WOT_E + (NL - 1) * WN_E;
  static constexpr int OFF_BLOB = 0;
  static constexpr int OFF_GROUPS = (BLOB_E * 2 + 127) & ~127;
  static constexpr int OFF_TAIL = OFF_GROUPS + G * GROUP_B;   // 2 KB of zeros: spill target of the last transposed view
  static constexpr int OFF_BARS = OFF_TAIL + 2048;
  static constexpr int OFF_CONST = OFF_BARS + 64;             // sd[8], inv[8], ls[8], kiv[8], kls[8]
  static constexpr int OFF_TMEM = OFF_CONST + 160;
  static constexpr int OFF_LOCK = OFF_TMEM + 16;              // int lock, int initialised[4] (SHARED)
  static constexpr int SMEM_BYTES = OFF_LOCK + 32;
  // ---- tensor memory, per group: D [H] | dW_2 .. dW_NL [H each] | dWo [16] | dW1T [16]
  //      SHARED: D of group 0 | D of group 1 | one set of accumulators
  static constexpr int TMEM_ACC = (NL - 1) * H + 32;
  static constexpr int TMEM_G = H + TMEM_ACC;
  static_assert((SHARED ? G * H + TMEM_ACC : G * TMEM_G) <= 512, "tensor memory");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
  static_assert(BLOB_E <= kTcBlobHalves, "operand blob scratch");
};

__host__ __device__ __forceinline__ int canon(int row, int k, int K_total) {
  return (row >> 3) * (K_total * 8) + (k >> 3) * 64 + (row & 7) * 8 + (k & 7);
}

// kind::f16, D fp32, A/B fp16, dense; a_mn / b_mn select MN-major operands (bits 15 / 16).
__host__ __device__ constexpr uint32_t idesc(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}


// fp32 master parameters of one net -> its fp16 operand images (canonical K-major).  off_w / off_b: [0] layer 1 (obs -> H),
// [l - 1] hidden layer l, [NL] output layer.
template <int H, int NL>
__global__ void pack_kernel(GradArgs A, __half* __restrict__ blob) {
  using S = Shape<H, NL>;     // (the operand images do not depend on the group arrangement)
  constexpr int KP = S::KP;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= S::BLOB_E) return;
  if (A.ctl != nullptr && A.ctl[0] != 0 && A.ctl[1] < A.iter) return;   // the policy loop has stopped (ml4ca_ppo_ctl)
  auto inv = [](int f, int K, int& row, int& k) {   // invert canon()
    const int rg = f / (K * 8), rem = f % (K * 8);
    row = rg * 8 + (rem % 64) / 8, k = (rem / 64) * 8 + rem % 8;
  };
  const float* P = A.params;
  float v = 0.f;
  int row, k, f = e;
  if (f < S::B1_E) {                               // B1 [j][k]: W1[k][j], b1[j] at k = obs
    inv(f, 16, row, k);
    if (k < A.obs) v = P[A.off_w[0] + k * H + row];
    else if (k == A.obs) v = P[A.off_b[0] + row];
  } else if ((f -= S::B1_E) < (NL - 1) * S::BH_E) { // B_l [j][k]: W_l[k][j], b_l[j] at k = H
    const int l = 1 + f / S::BH_E;                  // index into off_w / off_b
    inv(f % S::BH_E, KP, row, k);
    if (k < H) v = P[A.off_w[l] + k * H + row];
    else if (k == H) v = P[A.off_b[l] + row];
  } else if ((f -= (NL - 1) * S::BH_E) < S::BO_E) { // Bo [o][k]: Wo[k][o], bo[o] at k = H
    inv(f, KP, row, k);
    if (row < A.nout) {
      if (k < H) v = P[A.off_w[NL] + k * A.nout + row];
      else if (k == H) v = P[A.off_b[NL] + row];
    }
  } else if ((f -= S::BO_E) < S::WOT_E) {           // WoT [k][o]: Wo[k][o]
    inv(f, 16, row, k);
    if (k < A.nout) v = P[A.off_w[NL] + row * A.nout + k];
  } else {                                         // Wn_l [k_in][j]: W_l[k_in][j]
    f -= S::WOT_E;
    const int l = 1 + f / S::WN_E;
    inv(f % S::WN_E, H, row, k);
    v = P[A.off_w[l] + row * H + k];
  }
  blob[e] = __float2half_rn(v);
}

template <int ACTIVATION>
__device__ __forceinline__ uint32_t activate_pack(float lo, float hi) {
  const uint32_t x = pack_f16x2(lo, hi);
  uint32_t y;
  if constexpr (ACTIVATION == 1) {
    asm("{\n\t.reg .b32 t;\n\tmul.rn.f16x2 t, %1, %2;\n\tmax.f16x2 %0, %1, t;\n\t}" : "=r"(y) : "r"(x), "r"(0x32663266u));
  } else {
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(y) : "r"(x));
  }
  return y;
}
// f'(z) from the stored fp16 activation h = f(z)
template <int ACTIVATION>
__device__ __forceinline__ float2 act_grad2(uint32_t h2) {
  const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&h2));
  if constexpr (ACTIVATION == 1) return make_float2(h.x > 0.f ? 1.0f : 0.2f, h.y > 0.f ? 1.0f : 0.2f);
  return make_float2(1.0f - h.x * h.x, 1.0f - h.y * h.y);
}

// S97: the 9 -> 7 (pi) / 9 -> 1 (v) networks of RevoltFinal(extended_state, cont_ang) with the dims known at compile time.
template <int ACTIVATION, int NET, bool S97, int H, int NL, bool SH>
__global__ void __launch_bounds__((Shape<H, NL, SH>::THREADS), 1) ppo_grad_tc_kernel(const GradArgs A) {
  if (A.ctl != nullptr && A.ctl[0] != 0 && A.ctl[1] < A.iter) return;   // uniform: before any barrier / TMEM allocation
  using S = Shape<H, NL, SH>;
  constexpr int KP = S::KP, G = S::G, THREADS = S::THREADS, GROUP_B = S::GROUP_B, A0_B = S::A0_B, AH_B = S::AH_B, GO_B = S::GO_B;
  constexpr int OFF_BLOB = S::OFF_BLOB, OFF_GROUPS = S::OFF_GROUPS, OFF_BARS = S::OFF_BARS, OFF_CONST = S::OFF_CONST,
                OFF_TMEM = S::OFF_TMEM, BLOB_E = S::BLOB_E;
  extern __shared__ __align__(128) uint8_t smem[];
  // warp index through a shuffle: warp-uniform for the compiler, so the group index and every MMA descriptor derived from it
  // live in uniform registers (tcgen05.mma then issues back to back, without a per-thread waterfall loop)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  constexpr int SPLIT = S::SPLIT, GT = S::GT;
  const int g = warp / (4 * SPLIT), wg = warp % (4 * SPLIT);   // group, warp within the group
  const int half = wg >> 2, row = (wg & 3) * 32 + lane;        // which half of the columns (SPLIT = 2), sample row = TMEM lane
  const int c_lo = (SPLIT == 2 && half == 1) ? S::C_SPLIT : 0, c_hi = (SPLIT == 2 && half == 0) ? S::C_SPLIT : H;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BARS);
  float* consts = reinterpret_cast<float*>(smem + OFF_CONST);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_TMEM);
  const int obs = S97 ? 9 : A.obs, nout = S97 ? (NET == 0 ? 7 : 1) : A.nout, act_dim = S97 ? 7 : A.act;

  // ---- setup: operand images -> smem, zero the activation buffers, constant-1 columns, barriers, TMEM ------------------
  {
    const int4* src = reinterpret_cast<const int4*>(A.blob);
    int4* dst = reinterpret_cast<int4*>(smem + OFF_BLOB);
    for (int i = threadIdx.x; i < BLOB_E * 2 / 16; i += THREADS) dst[i] = src[i];
    int4* z = reinterpret_cast<int4*>(smem + OFF_GROUPS);
    for (int i = threadIdx.x; i < (G * GROUP_B + 2048) / 16; i += THREADS) z[i] = make_int4(0, 0, 0, 0);
    if (threadIdx.x < 8) {
      const int a = threadIdx.x;
      const float ls = (NET == 0 && a < nout) ? A.params[A.off_ls + a] : 0.f;
      const float sd = expf(ls);
      consts[a] = sd, consts[8 + a] = 1.0f / (sd + 1e-8f), consts[16 + a] = ls;
      const float lo = (NET == 0 && A.loss_mode == 1 && a < nout) ? A.kl_ls_old[a] : 0.f;        // trpo/core.py:57-58
      consts[24 + a] = 1.0f / (expf(2.0f * lo) + 1e-8f), consts[32 + a] = lo;
    }
  }
  __syncthreads();
  {
    uint8_t* base = smem + OFF_GROUPS + g * GROUP_B;
#pragma unroll
    for (int l = 1; l <= NL; ++l)                      // bias columns of the hidden operands
      reinterpret_cast<__half*>(base + A0_B + (l - 1) * AH_B)[canon(row, H, KP)] = __float2half_rn(1.0f);
  }
  if (threadIdx.x == 0) {
    for (int q = 0; q < 8; ++q) reinterpret_cast<int*>(smem + S::OFF_LOCK)[q] = 0;
    for (int q = 0; q < G; ++q) mbar_init(&bars[q], 2);   // the two issuing warps of a group each commit their part of a stage
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  // ---- per-group addresses ----------------------------------------------------------------------------------------------
  const uint32_t sb = smem_u32(smem);
  // operand buffers of the group: A0, A_l = activations leaving hidden layer l (l = 1 .. NL), G_out, one G_hidden buffer that
  // every back-propagated signal re-uses (its readers have completed before the next one is written: each epilogue waits)
  const uint32_t sA0 = sb + OFF_GROUPS + g * GROUP_B;
  auto sA = [&](int l) { return sA0 + A0_B + (uint32_t)(l - 1) * AH_B; };
  const uint32_t sGo = sA0 + A0_B + NL * AH_B, sGh = sGo + GO_B;       // (SHARED: no G_hidden buffer, sGh / pGh unused)
  // operand images: B1, B_l (l = 2 .. NL), Bo, WoT, Wn_l (l = 2 .. NL)
  const uint32_t sB1 = sb + OFF_BLOB;
  auto sB = [&](int l) { return sB1 + S::B1_E * 2 + (uint32_t)(l - 2) * S::BH_E * 2; };
  const uint32_t sBo = sB1 + S::B1_E * 2 + (NL - 1) * S::BH_E * 2, sWoT = sBo + S::BO_E * 2;
  auto sWn = [&](int l) { return sWoT + S::WOT_E * 2 + (uint32_t)(l - 2) * S::WN_E * 2; };
  uint8_t* gbase = smem + OFF_GROUPS + g * GROUP_B;
  __half* pA0 = reinterpret_cast<__half*>(gbase);
  auto pA = [&](int l) { return gbase + A0_B + (l - 1) * AH_B; };
  __half* pGo = reinterpret_cast<__half*>(gbase + A0_B + NL * AH_B);
  uint8_t* pGh = gbase + A0_B + NL * AH_B + GO_B;
  // accumulators: D, dW_l (l = 2 .. NL), dWo, dW1T
  constexpr bool SHARED = S::SHARED;
  const uint32_t tD = tmem_base + g * (SHARED ? H : S::TMEM_G);
  const uint32_t tAcc = SHARED ? tmem_base + G * H : tD + H;           // dW_2 .. dW_NL | dWo | dW1T
  const uint32_t tWo = tAcc + (NL - 1) * H, tW1 = tWo + 16;
  auto tW = [&](int l) { return tAcc + (uint32_t)(l - 2) * H; };
  int* lock = reinterpret_cast<int*>(smem + S::OFF_LOCK);             // [0] lock, [1 + a] accumulator a holds a tile already
  bool holds = false;                                                  // this group's weight-gradient chain is in flight under the lock
  const uint32_t lane_off = (uint32_t)((wg & 3) * 32) << 16;

  // MMA chains (one elected thread per group).  K-major operand: lbo = 128 B, sbo = K_total * 16 B, +256 B per k-step.
  // MN-major view of a buffer with K_total columns: lbo = K_total * 16 B, sbo = 128 B, + 2 lbo per k-step (16 samples).
  auto chain_k = [&](uint32_t d, uint32_t a, int ka, uint32_t b, int kb, int N, int steps, bool acc0) {
    const uint32_t id = idesc(128, N, 0, 0);
    for (int s = 0; s < steps; ++s)
      mma_f16(d, smem_desc(a + s * 256, 128, ka * 16), smem_desc(b + s * 256, 128, kb * 16), id, acc0 || s > 0);
  };
  auto chain_mn = [&](uint32_t d, uint32_t a, int ka, uint32_t b, int kb, int N, bool acc0) {
    const uint32_t id = idesc(128, N, 1, 1);
    for (int s = 0; s < 8; ++s)
      mma_f16(d, smem_desc(a + s * 2 * ka * 16, ka * 16, 128), smem_desc(b + s * 2 * kb * 16, kb * 16, 128), id, acc0 || s > 0);
  };
  uint32_t phase = 0;
  auto sync_group = [&]() {
    fence_async_smem();
    asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "n"(GT) : "memory");
  };
  auto wait_mma = [&]() {
    mbar_wait(&bars[g], phase);
    phase ^= 1;
    fence_after_sync();
    if constexpr (SHARED) {
      if (holds) {                             // group-uniform: the chain issued under the lock has completed
        if (wg == 0 && lane == 0) {
          fence_before_sync();
          __threadfence_block();
          atomicExch(lock, 0);
        }
        holds = false;
      }
    }
  };
  // weight-gradient chain into accumulator `a` (0 .. NL - 2: dW_2 .., NL - 1: dWo, NL: dW1T), called by the issuing lane.
  // Returns whether the accumulator holds a tile already (the first chain overwrites, the later ones accumulate).
  auto acc_begin = [&](int a, bool own_acc) -> bool {
    if constexpr (!SHARED) {
      return own_acc;
    } else {
      while (atomicCAS(lock, 0, 1) != 0) {
      }
      __threadfence_block();
      fence_after_sync();
      return atomicExch(&lock[1 + a], 1) != 0;
    }
  };

  const int64_t n = A.n;
  const int64_t total = n * (int64_t)A.T;       // tiles run over the flat sample index (common.h: split_sample)
  const int64_t num_tiles = (total + TS - 1) / TS;
  float dls[8];
#pragma unroll
  for (int a = 0; a < 8; ++a) dls[a] = 0.f;
  double st[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  bool acc = false, pending = false;   // acc: the dW accumulators hold a tile already; pending: the dW1T chain is in flight

  constexpr int kPreObs = S97 ? 9 : 12;        // observation rows fetched one tile ahead (wider inputs load the rest in place)
  float pf_o[kPreObs], pf_a[8], pf_adv = 0.f, pf_lpo = 0.f, pf_ret = 0.f;
  auto fetch = [&](int64_t tl) {
    const int64_t smp = tl * TS + row;
    const bool live = smp < total && half == 0;      // the second thread of a row takes no part in the inputs or the loss
    int64_t t = 0, i = 0;
    if (live) split_sample(smp, n, t, i);
#pragma unroll
    for (int c = 0; c < kPreObs; ++c) pf_o[c] = (c < obs && live) ? __ldg(A.obs_buf + ((int64_t)t * obs + c) * n + i) : 0.f;
#pragma unroll
    for (int a = 0; a < 8; ++a) pf_a[a] = 0.f;
    pf_adv = pf_lpo = pf_ret = 0.f;
    if constexpr (NET == 0) {
#pragma unroll
      for (int a = 0; a < 8; ++a)       // rows a mode does not use are NULL and read as zero (KL mode: act_buf = mu_old only)
        if (a < nout && live && A.act_buf != nullptr) pf_a[a] = __ldg(A.act_buf + ((int64_t)t * act_dim + a) * n + i);
      if (live && A.adv != nullptr) pf_adv = __ldg(A.adv + (int64_t)t * n + i);
      if (live && A.logp_old != nullptr) pf_lpo = __ldg(A.logp_old + (int64_t)t * n + i);
    } else {
      if (live) pf_ret = __ldg(A.ret + (int64_t)t * n + i);
    }
  };
  bool first_tile = true;
  // group g of CTA b takes tiles g * gridDim.x + b, + G gridDim.x, ...: with fewer tiles than CTAs x groups (the reference's own
  // batch: 4 x 400 samples = 13 tiles) every tile gets a CTA of its own and the other groups of that CTA stay idle
  for (int64_t tile = (int64_t)g * gridDim.x + blockIdx.x; tile < num_tiles; tile += (int64_t)gridDim.x * G) {
    const int64_t smp = tile * TS + row;
    const bool live = smp < total && half == 0;
    int64_t t = 0, i = 0;
    if (live) split_sample(smp, n, t, i);
    // ---- inputs: thread = sample.  Requested one tile ahead (below, after the first hand-over), so their HBM latency is
    // off the serial chain of the group; only the first tile loads in place.
    if (first_tile) {
      fetch(tile);
      first_tile = false;
    }
    float o[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) o[c] = (c < kPreObs) ? pf_o[c] : ((c < obs && live) ? __ldg(A.obs_buf + ((int64_t)t * obs + c) * n + i) : 0.f);
#pragma unroll
    for (int c = 0; c < 16; ++c)
      if (c == obs) o[c] = 1.0f;
    float av[8], adv = pf_adv, lpo = pf_lpo, ret = pf_ret;
#pragma unroll
    for (int a = 0; a < 8; ++a) av[a] = pf_a[a];
    if (pending) {                             // the previous tile's dW1T chain still reads A0 / G1
      wait_mma();
      pending = false;
    }
    if (half == 0) {
      uint32_t w[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) w[c] = pack_f16x2(o[2 * c], o[2 * c + 1]);
      *reinterpret_cast<uint4*>(pA0 + canon(row, 0, 16)) = make_uint4(w[0], w[1], w[2], w[3]);
      *reinterpret_cast<uint4*>(pA0 + canon(row, 8, 16)) = make_uint4(w[4], w[5], w[6], w[7]);
    }
    sync_group();
    if (wg < 2) {                                                  // warp-uniform: the two issuing warps of the group
      if (elect_one()) {
        fence_after_sync();
        if (wg == 0) {
          chain_k(tD, sA0, 16, sB1, 16, H, 1, false);              // F1
        }
        mma_commit(&bars[g]);
      }
      __syncwarp();
    }
    fetch(tile + (int64_t)gridDim.x * G);          // next tile's rows: AFTER the hand-over (its MEMBAR would wait for them)
    // ---- hidden epilogues: D -> f -> operand rows -------------------------------------------------------------------------
    auto hidden = [&](uint8_t* dst) {
      wait_mma();
      uint32_t buf[16];
#pragma unroll
      for (int c0 = 0; c0 < H; c0 += 16) {
        if (c0 < c_lo || c0 >= c_hi) continue;         // this thread's share of the row (warp-uniform)
        tmem_ld16_async(tD + lane_off + c0, buf);
        wait_ld();
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          uint32_t w[4];
#pragma unroll
          for (int k = 0; k < 4; ++k)
            w[k] = activate_pack<ACTIVATION>(__uint_as_float(buf[q * 8 + 2 * k]), __uint_as_float(buf[q * 8 + 2 * k + 1]));
          *reinterpret_cast<uint4*>(dst + (size_t)canon(row, c0 + q * 8, KP) * 2) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
      fence_before_sync();
      sync_group();
    };
#define ML4CA_ISSUE2(W0, W1)                                                                                      \
  if (wg < 2) { /* warp-uniform: the two issuing warps of the group */                                             \
    if (elect_one()) {                                                                                            \
      fence_after_sync();                                                                                         \
      if (wg == 0) {                                                                                              \
        W0;                                                                                                       \
      } else {                                                                                                    \
        W1;                                                                                                       \
      }                                                                                                           \
      mma_commit(&bars[g]);                                                                                       \
    }                                                                                                             \
    __syncwarp();                                                                                                 \
  }
#pragma unroll
    for (int l = 1; l <= NL; ++l) {
      hidden(pA(l));
      if (l < NL) {
        ML4CA_ISSUE2(chain_k(tD, sA(l), KP, sB(l + 1), KP, H, KP / 16, false), (void)0);       // F_{l+1}
      } else {
        ML4CA_ISSUE2(chain_k(tD, sA(NL), KP, sBo, KP, OP, KP / 16, false), (void)0);           // output layer
      }
    }
    // ---- loss: per-sample dOUT (sum convention), scaled, -> G_out ---------------------------------------------------------------
    wait_mma();
    float out[16];
    tmem_ld16(tD + lane_off, out);
    fence_before_sync();
    if (A.mu_out != nullptr) {                 // forward only (uniform): store the means of this tile, next tile
      if (live) {
#pragma unroll
        for (int a = 0; a < 8; ++a)
          if (a < nout) A.mu_out[((int64_t)t * nout + a) * n + i] = out[a];
      }
      continue;
    }
    float dout[8];
#pragma unroll
    for (int a = 0; a < 8; ++a) dout[a] = 0.f;
    if (NET == 0 && A.loss_mode == 1) {
      // d_kl = mean_s sum_a 0.5 (((mu_old - mu)^2 + var) / (var_old + EPS) - 1) + log_std_old - log_std  (trpo/core.py:52-60,98)
      double kl = 0.0;
#pragma unroll
      for (int a = 0; a < 8; ++a)
        if (a < nout) {
          const float d = out[a] - av[a], var = consts[a] * consts[a];
          kl += (double)(0.5f * ((d * d + var) * consts[24 + a] - 1.0f) + (consts[32 + a] - consts[16 + a]));
          dout[a] = live ? d * consts[24 + a] : 0.f;
          dls[a] += live ? (var * consts[24 + a] - 1.0f) : 0.f;
        }
      if (live) st[2] += kl;
    } else if constexpr (NET == 0) {
      float logp = 0.f, z[8];
#pragma unroll
      for (int a = 0; a < 8; ++a) {
        z[a] = 0.f;
        if (a < nout) {
          z[a] = (av[a] - out[a]) * consts[8 + a];                                  // core.py:45
          logp += -0.5f * (z[a] * z[a] + 2.0f * consts[16 + a] + 1.8378770664093453f);
        }
      }
      const float ratio = expf(logp - lpo);                                         // ppo.py:234
      const float min_adv = adv > 0.f ? (1.0f + A.clip) * adv : (1.0f - A.clip) * adv;
      const float ra = ratio * adv;
      const float dlogp = (live && ra <= min_adv) ? -ra : 0.f;
#pragma unroll
      for (int a = 0; a < 8; ++a)
        if (a < nout) {
          dout[a] = dlogp * z[a] * consts[8 + a];
          dls[a] += dlogp * (z[a] * z[a] * consts[a] * consts[8 + a] - 1.0f);
        }
      if (live) {
        st[0] += (double)fminf(ra, min_adv);
        const float dl = lpo - logp;
        st[2] += 0.5 * (double)dl * (double)dl;
        st[3] += (double)(-logp);
        st[4] += (ratio > 1.0f + A.clip || ratio < 1.0f - A.clip) ? 1.0 : 0.0;
      }
    } else {
      const float e = out[0] - ret;
      dout[0] = live ? 2.0f * e : 0.f;
      if (live) st[1] += (double)e * (double)e;
    }
    if (half == 0) {
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) w[k] = pack_f16x2(dout[2 * k] * kScale, dout[2 * k + 1] * kScale);
      *reinterpret_cast<uint4*>(pGo + canon(row, 0, 16)) = make_uint4(w[0], w[1], w[2], w[3]);
      *reinterpret_cast<uint4*>(pGo + canon(row, 8, 16)) = make_uint4(0u, 0u, 0u, 0u);
    }
    sync_group();
    ML4CA_ISSUE2(chain_mn(tWo, sA(NL), KP, sGo, 16, OP, acc_begin(NL - 1, acc)),   // dWo += A_NL^T G_out
                 chain_k(tD, sGo, 16, sWoT, 16, H, 1, false));                     // D = G_out WoT^T
    holds = SHARED;
    // ---- backward epilogues: G = D .* f'(h) ------------------------------------------------------------------------------------
    auto backward = [&](const uint8_t* hsrc, uint8_t* dst) {
      wait_mma();
      uint32_t buf[16];
#pragma unroll
      for (int c0 = 0; c0 < H; c0 += 16) {
        if (c0 < c_lo || c0 >= c_hi) continue;         // this thread's share of the row (warp-uniform)
        tmem_ld16_async(tD + lane_off + c0, buf);
        const uint4 h0 = *reinterpret_cast<const uint4*>(hsrc + (size_t)canon(row, c0, KP) * 2);
        const uint4 h1 = *reinterpret_cast<const uint4*>(hsrc + (size_t)canon(row, c0 + 8, KP) * 2);
        const uint32_t hh[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        wait_ld();
        uint32_t w[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float2 gr = act_grad2<ACTIVATION>(hh[k]);
          w[k] = pack_f16x2(__uint_as_float(buf[2 * k]) * gr.x, __uint_as_float(buf[2 * k + 1]) * gr.y);
        }
        constexpr int kDst = SHARED ? KP : H;
        *reinterpret_cast<uint4*>(dst + (size_t)canon(row, c0, kDst) * 2) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(dst + (size_t)canon(row, c0 + 8, kDst) * 2) = make_uint4(w[4], w[5], w[6], w[7]);
      }
      fence_before_sync();
      sync_group();
    };
#pragma unroll
    for (int l = NL; l >= 2; --l) {
      // G_l = D .* f'(A_l): into the G buffer (layout [128 x H]) or, SHARED, in place over A_l (layout [128 x KP])
      const uint32_t sG = SHARED ? sA(l) : sGh;
      constexpr int kG = SHARED ? KP : H;
      backward(pA(l), SHARED ? pA(l) : pGh);
      ML4CA_ISSUE2(chain_mn(tW(l), sA(l - 1), KP, sG, kG, H, acc_begin(l - 2, acc)),   // dW_l += A_{l-1}^T G_l
                   chain_k(tD, sG, kG, sWn(l), H, H, H / 16, false));                  // D = G_l Wn_l^T
      holds = SHARED;
    }
    {
      const uint32_t sG = SHARED ? sA(1) : sGh;
      constexpr int kG = SHARED ? KP : H;
      backward(pA(1), SHARED ? pA(1) : pGh);                         // G_1 (the buffer's readers have completed)
      ML4CA_ISSUE2(chain_mn(tW1, sG, kG, sA0, 16, OP, acc_begin(NL, acc)), (void)0);   // dW1T += G_1^T A0
      holds = SHARED;
    }
#undef ML4CA_ISSUE2
    acc = true;
    pending = true;                                                // waited for before A0 / G2 are written again
  }
  if (pending) wait_mma();

  // ---- flush: TMEM accumulators -> global gradient (one atomicAdd per element and group), statistics -------------------
  float* gr = A.grad;
  const float unscale = 1.0f / kScale;
  if constexpr (SHARED) {                      // one set of accumulators: flushed once both groups have finished, the groups
    fence_before_sync();                       // taking alternate 16-column chunks
    __syncthreads();
    fence_after_sync();
    acc = lock[1] != 0;                        // (every accumulator has been written once any tile went through the backward pass)
  }
  if (acc) {
    float v[16];
    // tcgen05.ld is warp-collective: every thread loads, the row test only guards the atomics
#pragma unroll
    for (int l = 2; l <= NL; ++l) {
#pragma unroll
      for (int c0 = 0; c0 < H; c0 += 16) {             // dW_l rows k = 0 .. H - 1, row H = bias b_l
        if (c0 < c_lo || c0 >= c_hi) continue;
        if (SHARED && ((c0 >> 4) % G) != g) continue;
        tmem_ld16(tW(l) + lane_off + c0, v);
        if (row <= H) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            atomicAdd(gr + (row < H ? A.off_w[l - 1] + row * H : A.off_b[l - 1]) + c0 + j, v[j] * unscale);
        }
      }
    }
    tmem_ld16(tWo + lane_off, v);
    if (row <= H && half == 0 && (!SHARED || g == 0)) {
#pragma unroll
      for (int o = 0; o < 8; ++o)
        if (o < nout) atomicAdd(gr + (row < H ? A.off_w[NL] + row * nout : A.off_b[NL]) + o, v[o] * unscale);
    }
    tmem_ld16(tW1 + lane_off, v);        // dW1T: lane = hidden unit j, column = input k (k = obs: bias b1)
    if (row < H && half == SPLIT - 1 && (!SHARED || g == G - 1)) {
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        if (k < obs) atomicAdd(gr + A.off_w[0] + k * H + row, v[k] * unscale);
        else if (k == obs) atomicAdd(gr + A.off_b[0] + row, v[k] * unscale);
      }
    }
  }
  fence_before_sync();
#pragma unroll
  for (int a = 0; a < 8; ++a) {
    float r = dls[a];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, off);
    if (NET == 0 && lane == 0 && a < nout && r != 0.f) atomicAdd(gr + A.off_ls + a, r);
  }
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    double r = st[q];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, off);
    if (lane == 0 && r != 0.0) atomicAdd(A.stats + q, r);
  }
  if (threadIdx.x == 0 && blockIdx.x == 0 && A.mu_out == nullptr) atomicAdd(A.stats + 5, (double)A.n * (double)A.T);
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

}  // namespace ppotc
}  // namespace ml4ca

using namespace ml4ca;

// Host side: called by grad_pass (ppo_update.cu) when the tensor-core switch of the pass is on.  `blob` is scratch for the
// packed fp16 operands (>= kTcBlobHalves halves), owned by the caller.
template <int H, int NL, bool SH = false>
static int launch_shape(const GradArgs& args, int activation, int net, void* blob, cudaStream_t st) {
  using S = ppotc::Shape<H, NL, SH>;
  GradArgs a = args;
  __half* b = static_cast<__half*>(blob);
  ppotc::pack_kernel<H, NL><<<(S::BLOB_E + 255) / 256, 256, 0, st>>>(a, b);
  int rc = check_launch("ppo pack_kernel");
  if (rc != ML4CA_OK) return rc;
  a.blob = b;
  const int64_t tiles = (a.n * (int64_t)a.T + ppotc::TS - 1) / ppotc::TS;
  const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
  const bool s97 = a.obs == 9 && a.act == 7;
  // the 9 -> 7 dims of RevoltFinal(extended_state, cont_ang) are compiled in; the other env classes (RevoltLimited: 5 actions,
  // RevoltSimple: 3, no extended state: 6 observations ...) take the instantiation with run-time dims
#define ML4CA_TC_LAUNCH(ACTV, NETV)                                                                                      \
  do {                                                                                                                   \
    auto k = ppotc::ppo_grad_tc_kernel<ACTV, NETV, true, H, NL, SH>;                                                     \
    if (!s97) k = ppotc::ppo_grad_tc_kernel<ACTV, NETV, false, H, NL, SH>;                                               \
    ML4CA_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, S::SMEM_BYTES));                     \
    k<<<grid, S::THREADS, S::SMEM_BYTES, st>>>(a);                                                                       \
  } while (0)
  if (activation == 1) {
    if (net == 0) ML4CA_TC_LAUNCH(1, 0); else ML4CA_TC_LAUNCH(1, 1);
  } else {
    if (net == 0) ML4CA_TC_LAUNCH(0, 0); else ML4CA_TC_LAUNCH(0, 1);
  }
#undef ML4CA_TC_LAUNCH
  return check_launch("ppo_grad_tc_kernel");
}

bool ml4ca_ppo_tc_supports(int hidden, int n_hidden, int obs, int act) {
  const bool shape = (hidden == 64 && (n_hidden == 2 || n_hidden == 3)) || (hidden == 80 && n_hidden == 3);   // what policy.cu runs forward
  return shape && obs >= 1 && obs <= 15 && act >= 1 && act <= 8;
}

int ml4ca_ppo_grad_tc_launch(const GradArgs& args, int activation, int net, void* blob, cudaStream_t st) {
  ML4CA_REQUIRE(ml4ca_ppo_tc_supports(args.hidden, args.n_hidden, args.obs, args.act), "shape not built for the tensor-core gradient kernel");
  if (args.hidden == 64) {
    if (args.n_hidden == 3) return launch_shape<64, 3>(args, activation, net, blob, st);
    return launch_shape<64, 2>(args, activation, net, blob, st);
  }
  // 80^3: the two-group kernel on shared accumulators streams large batches 1.4 x faster (5.1 against 3.65 G sample-passes/s), the
  // single-group kernel with two threads per row has the shorter launch (31 against 53 us for one wave of tiles: the reference's
  // own 4 x 400 batch)
  const int64_t tiles = (args.n * (int64_t)args.T + ppotc::TS - 1) / ppotc::TS;
  if (tiles > 2 * kNumSMs) return launch_shape<80, 3, true>(args, activation, net, blob, st);
  return launch_shape<80, 3, false>(args, activation, net, blob, st);
}
