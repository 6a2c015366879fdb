"""Philox4x32-10 counter-based RNG in NumPy, bit-identical to ml4ca_b200/csrc/philox.cuh.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference samples reset poses with NumPy's
global MT19937 (simtools.py:109-124); a serial generator cannot be shared by millions of
environments, so the build keys a counter RNG by (seed, global env id, episode, draw) and the
parity with the reference is distribution-level only (uniform on the same intervals).  The
oracle and the kernels, however, agree bit for bit.
"""
import numpy as np

_M0 = np.uint64(0xD2511F53)
_M1 = np.uint64(0xCD9E8D57)
_W0 = 0x9E3779B9
_W1 = 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10.  All inputs uint32 arrays (broadcastable); returns 4 uint32 arrays."""
    c0 = np.asarray(c0, dtype=np.uint64)
    c1 = np.asarray(c1, dtype=np.uint64)
    c2 = np.asarray(c2, dtype=np.uint64)
    c3 = np.asarray(c3, dtype=np.uint64)
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = int(k0) & 0xFFFFFFFF
    k1 = int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = _M0 * c0
        p1 = _M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0)) & _MASK, lo1, (hi0 ^ c3 ^ np.uint64(k1)) & _MASK, lo0
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return (c0.astype(np.uint32), c1.astype(np.uint32), c2.astype(np.uint32), c3.astype(np.uint32))


def symmetric_unit(x):
    """uint32 -> float32 in [-1, 1):  ((x >> 8) - 2^23) * 2^-23, exact in float32."""
    x = np.asarray(x, dtype=np.uint32)
    i = (x >> np.uint32(8)).astype(np.int64) - (1 << 23)
    return (i.astype(np.float32) * np.float32(2.0 ** -23)).astype(np.float32)


def unit_open(x):
    """uint32 -> float32 in (0, 1]:  ((x >> 8) + 1) * 2^-24 (used by Box-Muller, never 0)."""
    x = np.asarray(x, dtype=np.uint32)
    return ((x >> np.uint32(8)).astype(np.float32) + np.float32(1.0)) * np.float32(2.0 ** -24)


def symmetric_unit21(x):
    """low 21 bits -> float32 in [-1, 1):  ((x & 0x1FFFFF) - 2^20) * 2^-20, exact in float32."""
    i = (np.asarray(x, dtype=np.uint32) & np.uint32(0x1FFFFF)).astype(np.int64) - (1 << 20)
    return (i.astype(np.float32) * np.float32(2.0 ** -20)).astype(np.float32)


def reset_draws(seed, env_id, episode):
    """The six reset uniforms of one (env, episode word): ONE Philox block, counter (env_lo, env_hi, word, 0),
    split into six 21-bit fields: the low 21 bits of each of the four outputs, then the top 11 bits of
    outputs 0|1 and of outputs 2|3 (11 + 11 = 22 bits, masked to 21).

    Returns float32 array [6, n] of symmetric units in [-1, 1): N, E, psi, u, v, r order.
    Key = (seed_lo, seed_hi ^ 0x5EED5EED).
    """
    env_id = np.asarray(env_id, dtype=np.uint64)
    episode = np.asarray(episode, dtype=np.uint64)
    k0 = int(seed) & 0xFFFFFFFF
    k1 = ((int(seed) >> 32) & 0xFFFFFFFF) ^ 0x5EED5EED
    lo = env_id & _MASK
    hi = env_id >> np.uint64(32)
    q = philox4x32(lo, hi, episode & _MASK, np.zeros_like(lo), k0, k1)
    s = np.uint32
    v5 = (q[0] >> s(21)) | ((q[1] >> s(21)) << s(11))
    v6 = (q[2] >> s(21)) | ((q[3] >> s(21)) << s(11))
    return np.stack([symmetric_unit21(q[0]), symmetric_unit21(q[1]), symmetric_unit21(q[2]),
                     symmetric_unit21(q[3]), symmetric_unit21(v5), symmetric_unit21(v6)])


def reset_thrust_normals(seed, env_id, episode):
    """The three standard normals of a ``reset_acts`` restart (customEnv.py:181): SECOND Philox block of the
    (env, episode word), counter (env_lo, env_hi, word, 1); Box-Muller on (out0, out1) -> z0 = r cos, z1 = r sin and
    on (out2, out3) -> z2 = r cos, with r = sqrt(-2 ln unit_open(a)), angle = 2 pi (b >> 8) 2^-24.
    Same uniforms as csrc/env_math.cuh::sample_reset_thrust; evaluated in float64 here (the kernel's logf / sincospif
    are fp32, so agreement is ~1e-6 relative, not bit-level).  Returns float64 [3, n]."""
    env_id = np.asarray(env_id, dtype=np.uint64)
    episode = np.asarray(episode, dtype=np.uint64)
    k0 = int(seed) & 0xFFFFFFFF
    k1 = ((int(seed) >> 32) & 0xFFFFFFFF) ^ 0x5EED5EED
    lo = env_id & _MASK
    hi = env_id >> np.uint64(32)
    q = philox4x32(lo, hi, episode & _MASK, np.ones_like(lo), k0, k1)
    r0 = np.sqrt(-2.0 * np.log(unit_open(q[0]).astype(np.float64)))
    r1 = np.sqrt(-2.0 * np.log(unit_open(q[2]).astype(np.float64)))
    a0 = 2.0 * np.pi * (q[1] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    a1 = 2.0 * np.pi * (q[3] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    return np.stack([r0 * np.cos(a0), r0 * np.sin(a0), r1 * np.cos(a1)])


def policy_normals(seed, env_id, step):
    """The eight exploration normals of one (env, step) of the policy forward (csrc/policy.cu, policy_kernel): key
    (seed_lo, seed_hi ^ 0xAC710A), TWO Philox blocks with counters (id_lo, id_hi, step, 0) and (id_lo, id_hi, step, 1);
    Box-Muller on (x, y) and on (z, w) of each block -> eps[0..3] from the first block, eps[4..7] from the second, with
    r = sqrt(-2 ln unit_open(a)), angle = 2 pi (b >> 8) 2^-24, (r cos, r sin) per pair.  Evaluated in float64 (the kernel's
    __logf / __sincosf are fp32 approximations).  Returns float64 [8, n]; action a uses row a."""
    env_id = np.asarray(env_id, dtype=np.uint64)
    k0 = int(seed) & 0xFFFFFFFF
    k1 = ((int(seed) >> 32) & 0xFFFFFFFF) ^ 0xAC710A
    lo = env_id & _MASK
    hi = env_id >> np.uint64(32)
    st = np.full_like(lo, int(step) & 0xFFFFFFFF)
    out = []
    for block in (0, 1):
        q = philox4x32(lo, hi, st, np.full_like(lo, block), k0, k1)
        for a, b in ((q[0], q[1]), (q[2], q[3])):
            r = np.sqrt(-2.0 * np.log(unit_open(a).astype(np.float64)))
            ang = 2.0 * np.pi * (b >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
            out += [r * np.cos(ang), r * np.sin(ang)]
    return np.stack(out)
