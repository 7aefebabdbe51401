"""TEST INFRASTRUCTURE ONLY — NumPy restatement of the action samplers in csrc/rollout.cu (`sample_categorical_kernel`,
`sample_gaussian_kernel`) and float64 references of the operations they implement.  Not part of the product: only tests/ import
this module.

* `philox4x32_10`: Philox4x32-10 (Salmon et al. 2011, Random123's philox4x32 with 10 rounds), the kernel's round function and key
  schedule, vectorised over uint64 arrays that hold 32-bit words.
* `u01`: the kernel's word -> fp32 uniform, emulated exactly in float32: ((float)(x >> 8) + 0.5f) * 2^-24, clamped to the largest
  float below 1.  Every value lies in the open interval (0, 1).  The mapping is not uniform at the 2^-24 scale: for x >> 8 >= 2^23
  the sum needs 25 bits and rounds to even, so the upper half of the interval takes every other grid value, each twice as often.
* Stream layout.  Both kernels key Philox with the 64-bit seed (low word, high word) and count with (env lo, env hi, counter lo,
  counter hi), env = env_offset + row as a uint64 and counter = draw counter + device counter base (mod 2^64).  The categorical
  kernel reads word x of that counter.  The Gaussian kernel XORs `gaussian_pair_tag(p)` into the draw counter for dimension pair p
  and reads words x (radius) and y (angle) of Box-Muller.
* `categorical_reference` / `inverse_cdf`: float64 softmax, CDF and log_softmax of fp32 logits, and the inverse-CDF action of an
  exact uniform.  `gaussian_reference` / `normal_log_prob`: float64 Box-Muller from the exact fp32 uniforms of a draw,
  mean + exp(log_std) * n, and the Normal log-density of an action.
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
PHILOX_M0, PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
PHILOX_W0, PHILOX_W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
U01_MAX = np.float32(1.0) - np.float32(2.0 ** -24)          # 0x1.fffffep-1f, the largest float below 1
# seed 1, counter 0: the categorical word x of these environment ids has x >> 8 == 0xFFFFFF, the word that maps to U01_MAX
TOP_WORD_ENV_IDS = {8418514: 0xFFFFFF41, 27392119: 0xFFFFFFE4}


def _u64(x):
    return np.asarray(x, dtype=np.uint64)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counter (c0, c1, c2, c3) under key (k0, k1): 32-bit words in uint64 arrays (broadcast) -> (x, y, z, w)."""
    c0, c1, c2, c3, k0, k1 = (_u64(v) & M32 for v in (c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0, p1 = PHILOX_M0 * c0, PHILOX_M1 * c2                  # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + PHILOX_W0) & M32, (k1 + PHILOX_W1) & M32
    return c0, c1, c2, c3


def u01_unclamped(x):
    """((float)(x >> 8) + 0.5f) * 2^-24 in float32, as the samplers mapped words before the top word was clamped (it gives 1.0)."""
    return ((_u64(x) >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)


def u01(x):
    """The samplers' uniform of word x, bit-exact: in (0, 1)."""
    return np.minimum(u01_unclamped(x), U01_MAX)


def _words(seed, counter, env_ids):
    env = _u64(env_ids)
    counter = _u64(counter)
    seed = int(seed)
    return philox4x32_10(env & M32, env >> np.uint64(32), counter & M32, counter >> np.uint64(32), seed & 0xFFFFFFFF, seed >> 32)


def env_ids(env_offset, n):
    """Global environment ids env_offset + 0 .. n - 1 as the kernels form them (int64 sum, read as uint64)."""
    return (np.int64(env_offset) + np.arange(n, dtype=np.int64)).astype(np.uint64)


def draw_counter(counter, base=0):
    """Draw counter plus the device counter base, mod 2^64."""
    return np.uint64((int(counter) + int(base)) % (1 << 64))


def categorical_words(seed, counter, env_ids):
    """Word x of each environment's categorical draw."""
    return _words(seed, counter, env_ids)[0]


def gaussian_pair_tag(p):
    """Counter tag of dimension pair p: t = p + 1, low byte in bits 56-63, next byte in bits 48-55."""
    t = _u64(p) + np.uint64(1)
    return ((t & np.uint64(0xFF)) << np.uint64(56)) | ((t >> np.uint64(8)) << np.uint64(48))


def gaussian_pair_tag_unwidened(p):
    """(p + 1) << 56 mod 2^64: the tag before the second byte was added; 0 at p = 255, and p + 256 repeats p."""
    return (_u64(p) + np.uint64(1)) << np.uint64(56)


def gaussian_uniforms(seed, counter, env_ids, A):
    """Exact fp32 uniforms (u1 radius, u2 angle), each [N, A]: dimensions 2p and 2p + 1 share the draw of pair p."""
    P = (A + 1) // 2
    tags = gaussian_pair_tag(np.arange(P))
    x, y, _, _ = _words(seed, _u64(counter) ^ tags[None, :], _u64(env_ids)[:, None])
    return np.repeat(u01(x), 2, axis=1)[:, :A], np.repeat(u01(y), 2, axis=1)[:, :A]


def categorical_reference(logits):
    """float64 (softmax, CDF, log_softmax) of fp32 logits [N, A]; -inf entries get probability 0 (no row may be all -inf)."""
    z = np.asarray(logits, dtype=np.float64)
    mx = z.max(axis=1, keepdims=True)
    e = np.exp(z - mx)
    s = e.sum(axis=1, keepdims=True)
    return e / s, np.cumsum(e, axis=1) / s, z - mx - np.log(s)


def inverse_cdf(cdf, u):
    """The first action whose float64 CDF exceeds u (the last action for u at or above the row's total)."""
    a = (cdf <= np.asarray(u, dtype=np.float64)[:, None]).sum(axis=1)
    return np.minimum(a, cdf.shape[1] - 1)


def standard_normals(u1, u2):
    """float64 Box-Muller of the exact fp32 uniforms: even dimensions take the cosine, odd ones the sine."""
    u1, u2 = np.asarray(u1, dtype=np.float64), np.asarray(u2, dtype=np.float64)
    rad = np.sqrt(-2.0 * np.log(u1))
    ang = 2.0 * np.pi * u2
    odd = (np.arange(u1.shape[-1]) % 2).astype(bool)
    return rad, np.where(odd, rad * np.sin(ang), rad * np.cos(ang))


def gaussian_reference(mean, log_std, u1, u2):
    """float64 mean + exp(log_std) * n for the draw's uniforms; returns (actions, standard normals, Box-Muller radius)."""
    rad, n = standard_normals(u1, u2)
    return np.asarray(mean, np.float64) + np.exp(np.asarray(log_std, np.float64)) * n, n, rad


def normal_log_prob(actions, mean, log_std):
    """float64 sum over dimensions of log N(actions; mean, exp(log_std))."""
    a, m, ls = (np.asarray(v, dtype=np.float64) for v in (actions, mean, log_std))
    d = a - m
    return (-(d * d) / (2.0 * np.exp(2.0 * ls)) - ls - 0.5 * np.log(2.0 * np.pi)).sum(axis=-1)
