"""numpy Philox4x32-10 and the draw conventions shared with the CUDA kernels.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference has no
counter-based RNG (it draws from the global ``np.random`` state:
probayes/sp_utils.py:30-31, probayes/variable.py:631-633); this module defines
the *new* stream the device path uses so that a native-RNG device run can be
replayed bit-for-bit on the CPU via the injected-stream restatement.

Stream layout (must match probayes_b200/csrc/pbx_philox.cuh):
  key     = (seed & 0xffffffff, seed >> 32)
  counter = (step & 0xffffffff, step >> 32, chain, slot)
  slot s    : proposal draws for dims 2s, 2s+1 -- one block (w0..w3) per slot:
      u52 = (2*k + 1) * 2**-53,  k = (w0 << 20) | (w1 >> 12)        in (0, 1)
      u32 = (2*w2 + 1) * 2**-33                                     in (0, 1)
      normal pair : r = sqrt(-2 log u52), z0 = r cospi(2 u32), z1 = r sinpi(2 u32)
      uniform pair: (u52, u32)
  threshold : the spare bits of slot 0 -- t44 = (2*k + 1) * 2**-45,
      k = (w3 << 12) | (w1 & 0xfff)       => ONE Philox block per step for D <= 2
  (all three are exact in fp64 and strictly inside (0, 1))
  Gibbs (pbx_gibbs.cu): one uniform per global step g -- u52 of words (0, 1) (bit 2 of g
      clear) or (2, 3) (bit 2 set) of block (seed, g & ~4, chain, slot 0), so that steps g
      and g + 4 share a block
"""
import numpy as np

M0 = np.uint64(0xD2511F53)
M1 = np.uint64(0xCD9E8D57)
W0 = 0x9E3779B9
W1 = 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10. Inputs broadcastable integer arrays (< 2**32).
    Returns four uint64 arrays holding 32-bit words."""
    c0, c1, c2, c3 = np.broadcast_arrays(
        *[np.asarray(c, dtype=np.uint64) for c in (c0, c1, c2, c3)])
    c0, c1, c2, c3 = c0.copy(), c1.copy(), c2.copy(), c3.copy()
    k0 = int(k0) & 0xFFFFFFFF
    k1 = int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0
        p1 = M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0), lo1,
                          hi0 ^ c3 ^ np.uint64(k1), lo0)
        k0 = (k0 + W0) & 0xFFFFFFFF
        k1 = (k1 + W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def u52(w0, w1):
    """(2k+1)/2**53 with the 52-bit k = (w0 << 20) | (w1 >> 12)."""
    k = (w0 << np.uint64(20)) | (w1 >> np.uint64(12))
    return (2.0 * k.astype(np.float64) + 1.0) * 2.0 ** -53


def u32(w2):
    """(2 w2 + 1)/2**33."""
    return (2.0 * w2.astype(np.float64) + 1.0) * 2.0 ** -33


def t44(w3, w1):
    """(2k+1)/2**45 with the 44-bit k = (w3 << 12) | (w1 & 0xfff)."""
    k = (w3 << np.uint64(12)) | (w1 & np.uint64(0xFFF))
    return (2.0 * k.astype(np.float64) + 1.0) * 2.0 ** -45


def block(seed, step, chain, slot):
    seed = int(seed)
    step = np.asarray(step, dtype=np.uint64)
    return philox4x32_10(step & MASK, step >> np.uint64(32), chain, slot,
                         seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)


def uniform_pair(seed, step, chain, slot):
    w0, w1, w2, w3 = block(seed, step, chain, slot)
    return u52(w0, w1), u32(w2)


def normal_pair(seed, step, chain, slot):
    u1, u2 = uniform_pair(seed, step, chain, slot)
    r = np.sqrt(-2.0 * np.log(u1))
    # cospi/sinpi(2 u2); computed via exact-argument reduction to keep parity
    # with the device's sincospi to ~1 ulp
    return r * _cospi(2.0 * u2), r * _sinpi(2.0 * u2)


def _reduce_pi(x):
    # x in (0, 2): reduce to multiples of 0.5 exactly
    n = np.rint(2.0 * x)
    r = x - 0.5 * n           # exact, |r| <= 0.25
    return n.astype(np.int64) & 3, r * np.pi


def _sinpi(x):
    q, a = _reduce_pi(x)
    s, c = np.sin(a), np.cos(a)
    return np.choose(q, [s, c, -s, -c])


def _cospi(x):
    q, a = _reduce_pi(x)
    s, c = np.sin(a), np.cos(a)
    return np.choose(q, [c, -s, -c, s])


def normals(seed, steps, chains, ndim, step0=0):
    """Proposal normals Z[T, C, D] for steps step0..step0+T-1."""
    t = (np.arange(steps, dtype=np.uint64) + np.uint64(step0))[:, None]
    c = np.arange(chains, dtype=np.uint64)[None, :] if np.isscalar(chains) \
        else np.asarray(chains, dtype=np.uint64)[None, :]
    out = np.empty((steps, c.shape[1], ndim))
    for slot in range((ndim + 1) // 2):
        z0, z1 = normal_pair(seed, t, c, slot)
        out[:, :, 2 * slot] = z0
        if 2 * slot + 1 < ndim:
            out[:, :, 2 * slot + 1] = z1
    return out


def uniforms(seed, steps, chains, ndim, step0=0):
    """Proposal uniforms R[T, C, D] in (0,1) for steps step0..step0+T-1."""
    t = (np.arange(steps, dtype=np.uint64) + np.uint64(step0))[:, None]
    c = np.arange(chains, dtype=np.uint64)[None, :] if np.isscalar(chains) \
        else np.asarray(chains, dtype=np.uint64)[None, :]
    out = np.empty((steps, c.shape[1], ndim))
    for slot in range((ndim + 1) // 2):
        u0, u1 = uniform_pair(seed, t, c, slot)
        out[:, :, 2 * slot] = u0
        if 2 * slot + 1 < ndim:
            out[:, :, 2 * slot + 1] = u1
    return out


def spherical(seed, steps, chains, ndim, radius, scale=1.0, step0=0):
    """Spherical proposal deltas S[T, C, D] for steps step0..step0+T-1: the cube sample
    d = -r + 2r u (u as ``uniforms``) put on the sphere of radius r, ((d r) / |d|) * scale,
    with |d| from a sequential sum of squares (pbx_mh_mvn.cu draw_step, field.py:509-531).
    ``scale`` is a scalar or one factor per dimension."""
    d = -radius + (2.0 * radius) * uniforms(seed, steps, chains, ndim, step0)
    ss = np.zeros(d.shape[:-1])
    for j in range(ndim):
        ss = ss + d[..., j] * d[..., j]
    nrm = np.where(ss >= 2.2250738585072014e-308, np.sqrt(ss), 0.0)
    return ((d * radius) / nrm[..., None]) * np.broadcast_to(np.asarray(scale, float), (ndim,))


def thresholds(seed, steps, chains, step0=0):
    """Accept thresholds U[T, C]."""
    t = (np.arange(steps, dtype=np.uint64) + np.uint64(step0))[:, None]
    c = np.arange(chains, dtype=np.uint64)[None, :] if np.isscalar(chains) \
        else np.asarray(chains, dtype=np.uint64)[None, :]
    w0, w1, w2, w3 = block(seed, t, c, 0)
    return t44(w3, w1)


def gibbs_uniforms(seed, step, chain):
    """The Gibbs kernel's uniform for global step(s) ``step`` and chain id(s) ``chain``
    (broadcastable uint64 arrays): steps g and g + 4 share one Philox block."""
    step = np.asarray(step, dtype=np.uint64)
    w0, w1, w2, w3 = block(seed, step & ~np.uint64(4), chain, 0)
    return np.where((step & np.uint64(4)) != 0, u52(w2, w3), u52(w0, w1))
