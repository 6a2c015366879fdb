// philox.cuh -- Philox4x32-10 counter RNG (Salmon et al., SC'11), keyed by (seed, global env id, episode).
//
// Replaces the reference's NumPy global MT19937 reset sampling (specific/misc/simtools.py:109-124): a serial
// generator cannot be shared by millions of environments.  Parity with the reference is distribution-level
// (uniform on the same intervals); oracle/philox.py is bit-identical to this file.
#pragma once
#include <stdint.h>

namespace ml4ca {

// Counter = (env id lo, env id hi, episode word, tag): the tag (counter word 3) keeps the streams of one env and episode
// word apart.  Every new stream takes a tag no other stream uses.
constexpr uint32_t kTagResetPose = 0u;     // sample_reset: pose and velocity of a new episode
constexpr uint32_t kTagResetThrust = 1u;   // sample_reset_thrust: previous thrust of a new episode (reset_acts)
constexpr uint32_t kTagCurrent = 2u;       // sample_current: ocean current of a new episode (speed, direction)
constexpr uint32_t kTagBias0 = 3u;         // sample_disturbance: bias force of a new episode (stationary draw)
constexpr uint32_t kTagBiasStep = 4u;      // advance_bias: Gauss-Markov noise of one env step (word after the step)
constexpr uint32_t kTagWaveOmega = 5u;     // sample_waves: peak frequency of a new episode's wave motion (uniform, out0)
constexpr uint32_t kTagWaveMotion0 = 6u;   // sample_waves: stationary wave motion x of a new episode
constexpr uint32_t kTagWaveRate0 = 7u;     // sample_waves: stationary wave rate x' of a new episode
constexpr uint32_t kTagWaveStep1 = 8u;     // advance_waves: first normal of each DOF for one env step (word after the step)
constexpr uint32_t kTagWaveStep2 = 9u;     // advance_waves: second normal of each DOF for one env step

struct Philox4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return Philox4{c0, c1, c2, c3};
}

// uint32 -> float in [-1, 1): ((x >> 8) - 2^23) * 2^-23, exact in fp32.
__host__ __device__ __forceinline__ float symmetric_unit(uint32_t x) {
  return (float)((int32_t)(x >> 8) - (1 << 23)) * 1.1920928955078125e-07f;
}
// low 21 bits -> float in [-1, 1): ((x & 0x1FFFFF) - 2^20) * 2^-20, exact in fp32.
__host__ __device__ __forceinline__ float symmetric_unit21(uint32_t x) {
  return (float)((int32_t)(x & 0x1FFFFFu) - (1 << 20)) * 9.5367431640625e-07f;
}
// uint32 -> float in (0, 1]: ((x >> 8) + 1) * 2^-24.
__host__ __device__ __forceinline__ float unit_open(uint32_t x) {
  return ((float)(x >> 8) + 1.0f) * 5.9604644775390625e-08f;
}

}  // namespace ml4ca
