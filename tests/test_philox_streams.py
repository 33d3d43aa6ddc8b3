"""CPU checks of the numpy restatements of the device's Philox streams (oracle/philox.py): the classifier and
dynamics-fit noise layouts against an element-by-element restatement in plain Python integers, known answers, seed
truncation, and the hard-coded extreme counters the GPU tests in test_gpu_philox_draws.py rely on."""
import math

import numpy as np
import pytest

from oracle import philox as P

SEED_HI = (1 << 32) + 1234          # same low word as 1234: must give the same draws
# (row, block, word, x >> 9) for seed 1234, step 0 of the rollout noise stream: the ends of the uniform range.  At
# x >> 9 = 2^23 - 1, u = 1 - 2^-24 and the Box-Muller radius is 3.45e-4; at 0, u = 2^-24 and it is 5.77, the largest.
EXTREME_NOISE_WORDS = [(194945, 4, 0, (1 << 23) - 1), (1974695, 2, 0, (1 << 23) - 1), (3871307, 3, 0, (1 << 23) - 1),
                       (1489656, 1, 0, 0), (1564782, 1, 2, 0)]
EXTREME_SEED, EXTREME_STEP, EXTREME_S = 1234, 0, 17


def _philox_py(c, k):
    """Philox4x32-10 in Python integers (Salmon et al., SC'11)."""
    c, k0, k1 = list(c), k[0], k[1]
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k0) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, ((p0 >> 32) ^ c[3] ^ k1) & 0xFFFFFFFF, p0 & 0xFFFFFFFF]
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c


def _normal_py(words, w):
    """Word w of a block's Box-Muller pair, in float64: r cos t for even w, r sin t for odd w."""
    u = [((x >> 9) + 0.5) * 2.0 ** -23 for x in words]
    a = w & 2
    r, t = math.sqrt(-2.0 * math.log(u[a])), 2.0 * math.pi * u[a + 1]
    return r * (math.sin(t) if w & 1 else math.cos(t))


def _close(got, want):
    return abs(got - want) <= 2e-6 * (1.0 + abs(want))


@pytest.mark.parametrize("k,K", [(0, 2 * 17 + 6), (1, 17 + 6), (0, 2 * 2 + 1), (1, 3 + 2)])
def test_classifier_noise_layout(k, K):
    """Counter (row, k << 16 | j >> 2, draw, 0), key (seed, 'clsn'), word j & 3: every element of a few rows."""
    seed, draw, N = 99, 12, 7
    got = P.classifier_noise(seed, draw, N, K, k)
    assert got.shape == (N, K) and got.dtype == np.float32
    for i in (0, 3, N - 1):
        for j in range(K):
            words = _philox_py((i, (k << 16) | (j >> 2), draw, 0), (seed, P.STREAM_CLSN))
            assert _close(float(got[i, j]), _normal_py(words, j & 3)), (i, j)
    assert np.array_equal(P.classifier_noise(seed, draw, 2 * N, K, k)[:N], got)       # a row's noise does not depend on N


def test_classifier_noise_streams_are_distinct():
    """sas and sa never share noise, four columns never share a word, and each draw is fresh."""
    S, A, N, seed, draw = 17, 6, 64, 5, 3
    sas, sa = P.classifier_noise(seed, draw, N, 2 * S + A, 0), P.classifier_noise(seed, draw, N, S + A, 1)
    assert np.mean(sas[:, :S + A] == sa) < 0.01
    assert len({sas[:, j].tobytes() for j in range(2 * S + A)}) == 2 * S + A                # no two columns alike
    assert np.mean(P.classifier_noise(seed, draw + 1, N, 2 * S + A, 0) == sas) < 0.01
    assert abs(float(sas.mean())) < 0.05 and abs(float(sas.std()) - 1.0) < 0.05


@pytest.mark.parametrize("stream", [1, 2])
def test_fit_noise_layout(stream):
    """Counter (i >> 2 low, i >> 2 high, draw, stream), key (seed, 'fits'), word i & 3 of the block."""
    seed, draw, n = 31, 4, 6 * 7 * 3 * 16 + 3
    got = P.fit_noise(seed, draw, stream, n)
    assert got.shape == (n,) and got.dtype == np.float32
    for i in list(range(9)) + [n - 5, n - 1]:
        words = _philox_py((i >> 2, 0, draw, stream), (seed, P.STREAM_FIT))
        assert _close(float(got[i]), _normal_py(words, i & 3)), i
    assert np.array_equal(P.fit_noise(seed, draw, stream, 2 * n)[:n], got)               # a prefix of the longer stream
    assert np.mean(P.fit_noise(seed, draw, 3 - stream, n) == got) < 0.01


def test_rollout_noise_and_elite_slot_restated():
    """Rollout noise counter (row low, row high, step, block), key (seed, 'nois'); elite slot mulhi(x0, n_elites) with key
    (seed, 'elit'): rows past 2^32 and the last step word."""
    seed, step, S = 77, (1 << 32) - 1, 7
    rows = [0, (1 << 32) - 1, 1 << 32, (1 << 40) + 3]
    eps, slots, r = P.rollout_noise(seed, step, rows, S), P.rollout_elite_slot(seed, step, rows, 7), P.rollout_radius(seed, step, rows, S)
    for i, row in enumerate(rows):
        for j in range(S):
            words = _philox_py((row & 0xFFFFFFFF, row >> 32, step, j >> 2), (seed, P.STREAM_NOISE))
            assert _close(float(eps[i, j]), _normal_py(words, j & 3)), (row, j)
            ua = ((words[j & 2] >> 9) + 0.5) * 2.0 ** -23
            assert abs(r[i, j] - math.sqrt(-2.0 * math.log(ua))) <= 1e-12 * r[i, j] and abs(eps[i, j]) <= r[i, j] * (1 + 1e-6)
        x0 = _philox_py((row & 0xFFFFFFFF, row >> 32, step, 0), (seed, P.STREAM_ELITE))[0]
        assert slots[i] == (x0 * 7) >> 32
    assert not np.array_equal(eps[1], eps[2])                                             # the high row word is keyed


def test_known_answers():
    np.testing.assert_allclose(P.classifier_noise(7, 3, 3, 13, 0)[[0, 2], [1, 12]], [-2.6191769, -0.7010692], rtol=1e-6)
    np.testing.assert_allclose(P.classifier_noise(7, 3, 3, 9, 1)[[1, 2], [0, 8]], [0.92003435, 0.55421233], rtol=1e-6)
    np.testing.assert_allclose(P.fit_noise(7, 3, 1, 21)[[0, 5, 20]], [1.0593897, -1.1455406, 0.777124], rtol=1e-6)
    np.testing.assert_allclose(P.fit_noise(7, 3, 2, 21)[[0, 5, 20]], [0.28188545, -0.9461557, -1.8620492], rtol=1e-6)


def test_seed_truncated_to_low_word():
    rows = np.array([0, 5, (1 << 32) + 9])
    assert np.array_equal(P.rollout_noise(1234, 7, rows, 9), P.rollout_noise(SEED_HI, 7, rows, 9))
    assert np.array_equal(P.rollout_elite_slot(1234, 7, rows, 5), P.rollout_elite_slot(SEED_HI, 7, rows, 5))
    assert np.array_equal(P.classifier_noise(1234, 2, 5, 11, 1), P.classifier_noise(SEED_HI, 2, 5, 11, 1))
    assert np.array_equal(P.fit_noise(1234, 2, 2, 50), P.fit_noise(SEED_HI, 2, 2, 50))
    assert np.array_equal(P.buffer_indices(1234, 2, 50, 1000), P.buffer_indices(SEED_HI, 2, 50, 1000))
    assert not np.array_equal(P.rollout_noise(1234, 7, rows, 9), P.rollout_noise(1235, 7, rows, 9))


def test_extreme_counters_hit_the_ends_of_the_uniform_range():
    """The hard-coded counters of the GPU edge test really produce the extreme words, so that test cannot become vacuous."""
    key = np.array([EXTREME_SEED, P.STREAM_NOISE], np.uint32)
    rows = [c[0] for c in EXTREME_NOISE_WORDS]
    r = P.rollout_radius(EXTREME_SEED, EXTREME_STEP, rows, EXTREME_S)
    for i, (row, blk, w, top) in enumerate(EXTREME_NOISE_WORDS):
        assert 4 * blk + w < EXTREME_S
        out = P.philox4x32_10(np.array([row & 0xFFFFFFFF, row >> 32, EXTREME_STEP, blk], np.uint32), key)
        assert int(out[w]) >> 9 == top, (row, blk, w)
        want_r = math.sqrt(-2.0 * math.log(((top + 0.5) * 2.0 ** -23)))
        assert abs(r[i, 4 * blk + w] - want_r) <= 1e-9 * want_r
    assert r.min() < 3.5e-4 and r.max() > 5.76
