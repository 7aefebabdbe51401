"""CPU: the sampler restatement in tests/sampling_oracle.py -- Philox4x32-10 against Random123's known answers, the word -> uniform
mapping over every word class, the hard-coded environment ids whose first categorical word is a top word, and the Gaussian
dimension-pair tags.  The GPU tests (test_sampling_gpu.py) hold the kernels to this restatement."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sampling_oracle as SO  # noqa: E402


def _hex(words):
    return [f"{int(w):08x}" for w in words]


@pytest.mark.parametrize("ctr,key,expect", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, expect):
    """Random123's kat_vectors for philox4x32 with 10 rounds."""
    assert _hex(SO.philox4x32_10(*ctr, *key)) == expect.split()


def test_philox_vectorises_elementwise():
    c = np.arange(1000, dtype=np.uint64) * np.uint64(0x9E3779B1)
    x = SO.philox4x32_10(c & SO.M32, c >> np.uint64(16), np.uint64(7), np.uint64(3), 0x1234, 0xABCD)
    for i in (0, 1, 517, 999):
        one = SO.philox4x32_10(int(c[i]) & 0xFFFFFFFF, int(c[i]) >> 16, 7, 3, 0x1234, 0xABCD)
        assert [int(w[i]) for w in x] == [int(w) for w in one]


def test_uniform_is_inside_the_open_interval_for_every_word_class():
    """u01 depends on x >> 8 only: all 2^24 classes, at both ends of each class's low byte."""
    hi = np.arange(1 << 24, dtype=np.uint64)
    u = SO.u01(hi << np.uint64(8))
    assert u.dtype == np.float32
    assert np.array_equal(u.view(np.uint32), SO.u01((hi << np.uint64(8)) | np.uint64(0xFF)).view(np.uint32))
    assert u.min() > 0 and u.max() < 1
    assert u.min() == np.float32(2.0 ** -25) and u.max() == SO.U01_MAX
    assert np.all(np.diff(u) >= 0)                                           # monotone in the word


def test_uniform_keeps_every_value_but_the_top_word():
    hi = np.arange(1 << 24, dtype=np.uint64)
    old = SO.u01_unclamped(hi << np.uint64(8))
    new = SO.u01(hi << np.uint64(8))
    assert old[-1] == np.float32(1.0)                                        # 16777215.5f rounds to even: 2^24
    assert np.array_equal(new[:-1].view(np.uint32), old[:-1].view(np.uint32))
    assert new[-1].view(np.uint32) == np.uint32(0x3F7FFFFF)
    # the upper half rounds in pairs (documented, not corrected): k + 0.5 rounds to the even one of k, k + 1, so classes
    # 2^23 + 2j + 1 and 2^23 + 2j + 2 share the value (2^23 + 2j + 2) * 2^-24
    assert np.all(np.diff(new[:1 << 23]) > 0)
    up = new[(1 << 23) + 1:-1]
    assert np.array_equal(up[0::2], up[1::2]) and np.all(np.diff(up[0::2]) > 0)
    assert np.array_equal(up[1::2].astype(np.float64) * 2.0 ** 24, np.arange((1 << 23) + 2, 1 << 24, 2, dtype=np.float64))


def test_largest_uniform_times_any_row_sum_stays_below_it():
    """For every fp32 s in [1, 1024] (a categorical row's sum is at least 1 and at most A <= 1024), fl(u * s) < s at the largest
    u, hence for every u: the target of the inverse-CDF walk lies below the row's sum."""
    for e in range(10):
        bits = np.arange(np.float32(2.0 ** e).view(np.uint32), np.float32(2.0 ** (e + 1)).view(np.uint32), dtype=np.uint32)
        s = bits.view(np.float32)
        assert np.all(SO.U01_MAX * s < s), e
    assert SO.U01_MAX * np.float32(1024) < np.float32(1024)


def test_top_word_environment_ids():
    """Environment ids that draw the top word at seed 1, counter 0 (used by the GPU endpoint test)."""
    env = np.array(list(SO.TOP_WORD_ENV_IDS), dtype=np.uint64)
    x = SO.categorical_words(1, 0, env)
    assert [int(w) for w in x] == list(SO.TOP_WORD_ENV_IDS.values())
    assert np.all(x >= np.uint64(0xFFFFFF00))
    assert np.all(SO.u01_unclamped(x) == np.float32(1.0)) and np.all(SO.u01(x) == SO.U01_MAX)


def test_gaussian_pair_tags():
    p = np.arange(512)
    tags = SO.gaussian_pair_tag(p)
    assert np.all(tags != 0)                                                 # 0 is the categorical stream
    assert len(set(tags.tolist())) == 512                                    # A <= 1024 needs pairs 0..511
    assert np.all(tags & np.uint64((1 << 48) - 1) == 0)                      # draw counters below 2^48 cannot reach a tag
    assert np.array_equal(tags[:255], SO.gaussian_pair_tag_unwidened(p[:255]))
    old = SO.gaussian_pair_tag_unwidened(p)                                   # what the widened tag fixes
    assert old[255] == 0 and np.array_equal(old[256:], old[:256])
    assert len(set(SO.gaussian_pair_tag(np.arange(65535)).tolist())) == 65535


def test_gaussian_uniforms_follow_the_pair_layout():
    env = SO.env_ids((1 << 32) - 2, 4)
    u1, u2 = SO.gaussian_uniforms(5, 9, env, 7)
    assert u1.shape == u2.shape == (4, 7)
    for p in range(4):
        c = np.uint64(9) ^ SO.gaussian_pair_tag(p)
        x, y, _, _ = SO.philox4x32_10(env & SO.M32, env >> np.uint64(32), c & SO.M32, c >> np.uint64(32), 5, 0)
        for d in (2 * p, 2 * p + 1):
            if d < 7:
                assert np.array_equal(u1[:, d], SO.u01(x)) and np.array_equal(u2[:, d], SO.u01(y))


def test_categorical_reference():
    z = np.array([[0.0, np.log(3.0), -np.inf], [-np.inf, 5.0, -np.inf]], dtype=np.float32)
    p, cdf, lsm = SO.categorical_reference(z)
    np.testing.assert_allclose(p, [[0.25, 0.75, 0.0], [0.0, 1.0, 0.0]], rtol=1e-7)
    np.testing.assert_allclose(cdf[:, -1], 1.0, rtol=1e-15)
    np.testing.assert_allclose(lsm[0, :2], np.log([0.25, 0.75]), rtol=1e-7)
    assert lsm[0, 2] == -np.inf and lsm[1, 1] == 0.0
    assert SO.inverse_cdf(cdf, np.array([0.2499, 0.9])).tolist() == [0, 1]
    assert SO.inverse_cdf(cdf, np.array([0.25, 0.0])).tolist() == [1, 1]
    assert SO.inverse_cdf(cdf[:1, :2], np.array([1.0])).tolist() == [1]


def test_gaussian_reference():
    u1 = np.array([[np.exp(-0.5), np.exp(-0.5), np.exp(-2.0)]], dtype=np.float64)
    u2 = np.array([[0.25, 0.25, 0.5]])
    a, n, rad = SO.gaussian_reference(np.array([[1.0, 2.0, 3.0]]), np.array([0.0, np.log(2.0), 0.0]), u1, u2)
    np.testing.assert_allclose(rad, [[1.0, 1.0, 2.0]], rtol=1e-15)
    np.testing.assert_allclose(n, [[0.0, 1.0, -2.0]], atol=1e-15)
    np.testing.assert_allclose(a, [[1.0, 4.0, 1.0]], atol=1e-15)
    lp = SO.normal_log_prob(a, [[1.0, 2.0, 3.0]], np.array([0.0, np.log(2.0), 0.0]))
    np.testing.assert_allclose(lp, [-0.5 - 2.0 - np.log(2.0) - 1.5 * np.log(2 * np.pi)], rtol=1e-14)
