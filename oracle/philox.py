"""Philox4x32-10 counter RNG in numpy (oracle for csrc/philox.cuh).

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference draws its noise
from torch's global generator and NumPy's global RNG
(algo/dynamics/mobody_dynamics.py:220,225; algo/utils.py:128), which cannot be
reproduced on a device or across GPU counts.  The product's *production* mode
therefore uses Philox4x32-10 (Salmon et al., SC'11, the published Random123
algorithm) keyed on (seed, stream) with the counter holding (global_row, step,
block) so results do not depend on how rows are sharded.  This file restates
that published algorithm so the CUDA generator can be checked bit-for-bit.

Only the low 32 bits of a seed key the generator (``seed & 0xFFFFFFFF`` here,
``(uint32_t)seed`` on the device): seeds that differ by a multiple of 2^32 give
the same draws.

It also defines ``recipe_fill``: a torch-RNG-independent way to fill weight
tensors, so golden fixtures can name a recipe instead of storing megabytes.
"""
import numpy as np

_M0 = np.uint64(0xD2511F53)
_M1 = np.uint64(0xCD9E8D57)
_W0 = np.uint32(0x9E3779B9)
_W1 = np.uint32(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: uint32[..., 4], key: uint32[..., 2] (broadcastable) -> uint32[..., 4]."""
    ctr = np.asarray(ctr, dtype=np.uint32)
    key = np.asarray(key, dtype=np.uint32)
    c0, c1, c2, c3 = (ctr[..., i].astype(np.uint64) for i in range(4))
    shape = np.broadcast(c0, key[..., 0]).shape
    k0 = np.broadcast_to(key[..., 0], shape).astype(np.uint32)
    k1 = np.broadcast_to(key[..., 1], shape).astype(np.uint32)
    with np.errstate(over="ignore"):
        for r in range(10):
            p0 = _M0 * c0
            p1 = _M1 * c2
            hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
            hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
            n0 = hi1 ^ c1 ^ k0.astype(np.uint64)
            n2 = hi0 ^ c3 ^ k1.astype(np.uint64)
            c0, c1, c2, c3 = n0, lo1, n2, lo0
            if r != 9:
                k0 = (k0 + _W0).astype(np.uint32)
                k1 = (k1 + _W1).astype(np.uint32)
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def philox_uniform(bits):
    """uint32 -> fp32 in (0,1): ((x>>9)+0.5)*2^-23, exact in fp32."""
    x = (np.asarray(bits, dtype=np.uint32) >> np.uint32(9)).astype(np.float32)
    return (x + np.float32(0.5)) * np.float32(2.0 ** -23)


def philox_normal_pairs(bits4):
    """uint32[...,4] -> fp32[...,4] standard normals by Box-Muller.

    (x0,x1) -> (r cos t, r sin t), (x2,x3) likewise, with r=sqrt(-2 ln u_even),
    t = 2*pi*u_odd.  fp32 throughout, like the device code.
    """
    u = philox_uniform(bits4)
    out = np.empty(u.shape, dtype=np.float32)
    two_pi = np.float32(6.283185307179586)
    for a in (0, 2):
        r = np.sqrt(np.float32(-2.0) * np.log(u[..., a]), dtype=np.float32)
        t = two_pi * u[..., a + 1]
        out[..., a] = r * np.cos(t, dtype=np.float32)
        out[..., a + 1] = r * np.sin(t, dtype=np.float32)
    return out


# ---- production-mode draws used by the rollout (mirrors csrc/philox.cuh) ----
STREAM_NOISE = 0x6E6F6973  # 'nois'
STREAM_ELITE = 0x656C6974  # 'elit'
STREAM_INDEX = 0x696E6478  # 'indx'


def rollout_noise(seed, step, rows, S):
    """eps[len(rows), S] for the *picked* member of each global row.

    counter = (row_lo, row_hi, step, block), key = (seed, STREAM_NOISE);
    block b yields dims 4b..4b+3.
    """
    rows = np.asarray(rows, dtype=np.uint64)
    nb = (S + 3) // 4
    ctr = np.zeros((len(rows), nb, 4), dtype=np.uint32)
    ctr[..., 0] = (rows & np.uint64(0xFFFFFFFF)).astype(np.uint32)[:, None]
    ctr[..., 1] = (rows >> np.uint64(32)).astype(np.uint32)[:, None]
    ctr[..., 2] = np.uint32(step)
    ctr[..., 3] = np.arange(nb, dtype=np.uint32)[None, :]
    key = np.array([seed & 0xFFFFFFFF, STREAM_NOISE], dtype=np.uint32)
    n = philox_normal_pairs(philox4x32_10(ctr, key)).reshape(len(rows), nb * 4)
    return n[:, :S].copy()


def rollout_radius(seed, step, rows, S):
    """r[len(rows), S]: the Box-Muller radius sqrt(-2 ln u) of the pair each entry of rollout_noise() belongs to
    (|noise| <= r; errors of a device sine / cosine scale with r, not with the sample)."""
    rows = np.asarray(rows, dtype=np.uint64)
    nb = (S + 3) // 4
    ctr = np.zeros((len(rows), nb, 4), dtype=np.uint32)
    ctr[..., 0] = (rows & np.uint64(0xFFFFFFFF)).astype(np.uint32)[:, None]
    ctr[..., 1] = (rows >> np.uint64(32)).astype(np.uint32)[:, None]
    ctr[..., 2] = np.uint32(step)
    ctr[..., 3] = np.arange(nb, dtype=np.uint32)[None, :]
    key = np.array([seed & 0xFFFFFFFF, STREAM_NOISE], dtype=np.uint32)
    u = philox_uniform(philox4x32_10(ctr, key)).astype(np.float64)
    r = np.sqrt(-2.0 * np.log(u[..., [0, 0, 2, 2]]))
    return r.reshape(len(rows), nb * 4)[:, :S].copy()


def rollout_elite_slot(seed, step, rows, n_elites):
    """slot[len(rows)] in [0, n_elites): mulhi(x0, n_elites) (unbiased enough, no modulo)."""
    rows = np.asarray(rows, dtype=np.uint64)
    ctr = np.zeros((len(rows), 4), dtype=np.uint32)
    ctr[:, 0] = (rows & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    ctr[:, 1] = (rows >> np.uint64(32)).astype(np.uint32)
    ctr[:, 2] = np.uint32(step)
    key = np.array([seed & 0xFFFFFFFF, STREAM_ELITE], dtype=np.uint32)
    x0 = philox4x32_10(ctr, key)[:, 0].astype(np.uint64)
    return ((x0 * np.uint64(n_elites)) >> np.uint64(32)).astype(np.int64)


def buffer_indices(seed, draw, n, size):
    """int64[n] uniform in [0,size): replacement for np.random.randint in ReplayBuffer.sample.

    counter = (i_lo, i_hi, draw, 0), key = (seed, STREAM_INDEX); index = mulhi64(x0|x1<<32, size).
    """
    i = np.arange(n, dtype=np.uint64)
    ctr = np.zeros((n, 4), dtype=np.uint32)
    ctr[:, 0] = (i & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    ctr[:, 1] = (i >> np.uint64(32)).astype(np.uint32)
    ctr[:, 2] = np.uint32(draw)
    key = np.array([seed & 0xFFFFFFFF, STREAM_INDEX], dtype=np.uint32)
    out = philox4x32_10(ctr, key)
    # 64x64->hi64 via python ints would be slow; size < 2^32 in practice so use
    # the 32-bit form: (x0 * size) >> 32, identical to the device code.
    assert size < (1 << 32)
    return ((out[:, 0].astype(np.uint64) * np.uint64(size)) >> np.uint64(32)).astype(np.int64)


# ---- noise of the update kernels (mirrors csrc/train.cu and csrc/dynfit.cu) ----
STREAM_CLSN = 0x636C736E  # 'clsn'
STREAM_FIT = 0x66697473   # 'fits'


def classifier_noise(seed, draw, N, K, k):
    """randn_like of the classifier inputs: fp32[N, K] for batch rows 0..N-1 of classifier k (0: sas with K = 2S+A,
    1: sa with K = S+A).  Element (i, j) is word j & 3 of the Box-Muller block of counter (i, k << 16 | j >> 2, draw, 0),
    key (seed, STREAM_CLSN): the two classifiers never share a counter."""
    nb = (K + 3) // 4
    ctr = np.zeros((N, nb, 4), dtype=np.uint32)
    ctr[..., 0] = np.arange(N, dtype=np.uint32)[:, None]
    ctr[..., 1] = (np.uint32(k) << np.uint32(16)) | np.arange(nb, dtype=np.uint32)[None, :]
    ctr[..., 2] = np.uint32(draw)
    key = np.array([seed & 0xFFFFFFFF, STREAM_CLSN], dtype=np.uint32)
    return philox_normal_pairs(philox4x32_10(ctr, key)).reshape(N, nb * 4)[:, :K].copy()


def fit_noise(seed, draw, stream, n):
    """fp32[n]: element i of the dynamics-fit noise stream (1: the six reparameterised latents, flattened [6,7,B,16];
    2: the next-state noise, flattened [7,B,S]).  Element i is word i & 3 of the Box-Muller block of counter
    (i >> 2 low, i >> 2 high, draw, stream), key (seed, STREAM_FIT)."""
    nb = (n + 3) // 4
    blk = np.arange(nb, dtype=np.uint64)
    ctr = np.zeros((nb, 4), dtype=np.uint32)
    ctr[:, 0] = (blk & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    ctr[:, 1] = (blk >> np.uint64(32)).astype(np.uint32)
    ctr[:, 2] = np.uint32(draw)
    ctr[:, 3] = np.uint32(stream)
    key = np.array([seed & 0xFFFFFFFF, STREAM_FIT], dtype=np.uint32)
    return philox_normal_pairs(philox4x32_10(ctr, key)).reshape(-1)[:n].copy()


def recipe_fill(shape, seed, scale):
    """Deterministic fp32 fill: uniform in (-scale*sqrt3, scale*sqrt3) (std == scale).

    Element i uses word (i % 4) of philox4x32_10(ctr=(i//4,0,0,0), key=(seed, 0x77676874)).
    Independent of torch/numpy RNG implementations, so fixtures can store the
    recipe (seed, scale) instead of the weights.
    """
    n = int(np.prod(shape))
    nb = (n + 3) // 4
    ctr = np.zeros((nb, 4), dtype=np.uint32)
    ctr[:, 0] = np.arange(nb, dtype=np.uint32)
    key = np.array([seed & 0xFFFFFFFF, 0x77676874], dtype=np.uint32)
    u = philox_uniform(philox4x32_10(ctr, key)).reshape(-1)[:n]
    w = (np.float32(2.0) * u - np.float32(1.0)) * np.float32(scale * 3.0 ** 0.5)
    return w.astype(np.float32).reshape(shape)
