"""TEST INFRASTRUCTURE ONLY -- Philox-4x32-10 and the two uniform conversions of
``rlzero_b200/csrc/rz_common.cuh:172-203``, restated line for line.

The device draws every random number that decides a search's backed-up values from this generator
(random playouts, the child-order keys).  All of it is integer arithmetic, so the restatement
reproduces the device draws bit for bit; it is pinned to the published Random123 known-answer vectors
by ``tests/test_oracle_philox.py``.

``philox4`` works on Python ints (one counter); ``philox4_np`` on numpy arrays (many counters at once,
uint64 lanes masked to 32 bits so that no product overflows).
"""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57          # rz_philox_round multipliers
W0, W1 = 0x9E3779B9, 0xBB67AE85          # key schedule (Weyl) constants
MASK32 = 0xFFFFFFFF


def philox4(c0, c1, c2, c3, seed):
    """rz_philox4 (rz_common.cuh:185-195): the four 32-bit words for counter (c0..c3) and the 64-bit
    key ``seed`` (low word k0, high word k1).  Arguments are reduced to their low 32 / 64 bits like the
    device's ``uint32_t`` / ``unsigned long long`` parameters."""
    c = [c0 & MASK32, c1 & MASK32, c2 & MASK32, c3 & MASK32]
    seed &= (1 << 64) - 1
    k0, k1 = seed & MASK32, seed >> 32
    for _ in range(10):
        p0 = M0 * c[0]                    # rz_philox_round (rz_common.cuh:178-184)
        p1 = M1 * c[2]
        hi0, lo0 = p0 >> 32, p0 & MASK32
        hi1, lo1 = p1 >> 32, p1 & MASK32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + W0) & MASK32
        k1 = (k1 + W1) & MASK32
    return tuple(c)


def philox4_np(c0, c1, c2, c3, seed):
    """``philox4`` over arrays: the counters broadcast against each other, ``seed`` is one Python int or
    an array of uint64.  Returns a (4, ...) uint32 array."""
    u = np.uint64
    m32 = u(MASK32)
    c = [np.asarray(x, dtype=np.int64).astype(u) & m32 for x in (c0, c1, c2, c3)]
    c = list(np.broadcast_arrays(*c))
    if isinstance(seed, (int, np.integer)):
        seed = int(seed) & ((1 << 64) - 1)
        k0 = np.full(c[0].shape, seed & MASK32, dtype=u)
        k1 = np.full(c[0].shape, seed >> 32, dtype=u)
    else:
        s = np.broadcast_to(np.asarray(seed, dtype=u), c[0].shape)
        k0, k1 = s & m32, s >> u(32)
    for _ in range(10):
        p0 = u(M0) * c[0]                 # < 2^64: both factors are below 2^32
        p1 = u(M1) * c[2]
        hi0, lo0 = p0 >> u(32), p0 & m32
        hi1, lo1 = p1 >> u(32), p1 & m32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + u(W0)) & m32
        k1 = (k1 + u(W1)) & m32
    return np.stack(c).astype(np.uint32)


def u01_53(a, b):
    """rz_u01_53 (rz_common.cuh:197-200): uniform in (0, 1) from 53 bits of (a << 32 | b), float64."""
    x = (((a & MASK32) << 32) | (b & MASK32)) >> 11
    return (float(x) + 0.5) * (1.0 / 9007199254740992.0)


def u01_24(a):
    """rz_u01_24 (rz_common.cuh:201-203): uniform in (0, 1) from the top 24 bits of a, float32."""
    return (np.float32((a & MASK32) >> 8) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)


def pick(word, n):
    """``(rnd * n) >> 32``: the index in [0, n) the playout kernels draw from one Philox word."""
    return ((word & MASK32) * n) >> 32
