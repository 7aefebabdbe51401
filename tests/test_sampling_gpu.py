"""GPU: dppo_sample_categorical and dppo_sample_gaussian draw by draw against the float64 references of tests/sampling_oracle.py,
which restates their Philox4x32-10 streams bit for bit: the chosen action's CDF interval and log-prob, the Gaussian action and
log-prob, the draws that meet the top word, more than 512 action dimensions, the device counter base, and launch-shape
independence.  Every tolerance is a worst-case fp32 error bound derived in the helper that computes it."""
import itertools
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sampling_oracle as SO  # noqa: E402

EPS = 2.0 ** -24                                    # unit roundoff of fp32 round-to-nearest
SEEDS = (1, (1 << 40) + 3)                          # the second one fills the key's high word
COUNTERS = (0, (1 << 33) + 5)                       # the second one fills counter word 3
OFFSETS = (0, (1 << 32) - 70)                       # environment ids straddle 2^32 (counter word 1) at N > 70
STREAMS = list(itertools.product(SEEDS, COUNTERS, OFFSETS))
TWO_PI_F32 = float(np.float32(2.0 * np.pi))


@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as N
    return N.get_context(0)


def _cuda(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x)).to(device="cuda", dtype=dtype)


def _sample_categorical(ctx, logits_dev, seed, counter, env_offset):
    lp = torch.empty(logits_dev.shape[0], device="cuda")
    a = ctx.sample_categorical(logits_dev, seed, counter, env_offset, log_probs=lp)
    return a.cpu().numpy(), lp.cpu().numpy()


def _sample_gaussian(ctx, mean_dev, log_std_dev, seed, counter, env_offset):
    lp = torch.empty(mean_dev.shape[0], device="cuda")
    a = ctx.sample_gaussian(mean_dev, log_std_dev, seed, counter, env_offset, log_probs=lp)
    return a.cpu().numpy(), lp.cpu().numpy()


# ---------------------------------------------------------------- categorical -------------------------
def cdf_band(A):
    """Bound on |cum_j / s - C_j| + |target / s - u| for the kernel's fp32 walk, as a fraction of the row's sum (C: float64 CDF).

    Terms e_j = expf(fl(z_j - mx)): the subtraction's rounding moves exp(d) (d <= 0) by at most |d| e^d EPS <= EPS / e absolutely,
    and expf is within 2 ulp (4 EPS relative); the row's sum is at least 1, so both are relative to it.  cum_j and s are
    recursive fp32 sums of non-negative terms, each within (A - 1) EPS of its exact value relative to the full sum.  cum_j / s then
    differs from C_j by at most 2 ((A - 1) + 4 + A / e) EPS, and target = fl(u s) adds EPS: (2.74 A + 7) EPS, rounded up to cover
    second-order terms."""
    return (3 * A + 8) * EPS


def log_prob_bound(A, mx, log_s, lp_ref):
    """Bound on |logp - log_softmax| for logp = fl(z_a - fl(mx + logf(s))): s is within (A - 1 + 4 + A / e) EPS of its exact value
    (see cdf_band), which moves log s by as much absolutely; logf adds 1 ulp (2 EPS |log s|); the two roundings add EPS |mx + log s|
    and EPS |logp|.  Rounded up to (2 A + 4) for the sum and one more EPS for second-order terms."""
    return EPS * (2 * A + 5 + 2 * log_s + np.abs(mx) + log_s + np.abs(lp_ref))


def categorical_logits(rng, N, A):
    """Rows cycle through eight regimes: randn * {1e-3, 1, 30}; 1e4 + randn (mx + logf(s) in fp32); -inf at the first, a middle and
    the last action (A > 1); every action but one -inf."""
    z = rng.standard_normal((N, A))
    regime = np.arange(N) % 8
    z[regime == 0] *= 1e-3
    z[regime == 2] *= 30.0
    z[regime == 3] += 1e4
    if A > 1:
        z[regime == 4, 0] = -np.inf
        z[regime == 5, A // 2] = -np.inf
        z[regime == 6, A - 1] = -np.inf
    rows = np.flatnonzero(regime == 7)
    keep = rng.integers(0, A, rows.size)
    z[rows] = -np.inf
    z[rows, keep] = rng.standard_normal(rows.size)
    return z.astype(np.float32)


def check_categorical_draws(z, actions, lp, u, exact_share=None):
    """Every draw of rows z against float64: non-zero probability, u inside the action's CDF interval widened by cdf_band, the
    log-prob within log_prob_bound, and (exact_share) at least that share of draws equal to the float64 inverse-CDF action."""
    N, A = z.shape
    p, cdf, lsm = SO.categorical_reference(z)
    rows = np.arange(N)
    assert actions.dtype == np.int64 and np.all((actions >= 0) & (actions < A))
    zero = p[rows, actions] == 0
    assert not zero.any(), f"zero-probability actions at rows {np.flatnonzero(zero)[:8]} (u = {u[zero][:8]})"
    lo = np.where(actions > 0, cdf[rows, np.maximum(actions - 1, 0)], 0.0)
    hi = cdf[rows, actions]
    band = cdf_band(A)
    out = (u < lo - band) | (u > hi + band)
    assert not out.any(), (np.flatnonzero(out)[:8], u[out][:8], lo[out][:8], hi[out][:8])
    ref_lp = lsm[rows, actions]
    z64 = z.astype(np.float64)
    mx = z64.max(axis=1)
    log_s = np.log(np.exp(z64 - mx[:, None]).sum(axis=1))
    err = np.abs(lp.astype(np.float64) - ref_lp)
    bound = log_prob_bound(A, mx, log_s, ref_lp)
    assert np.all(np.isfinite(lp)) and np.all(err <= bound), (np.flatnonzero(err > bound)[:8], (err / bound).max())
    if exact_share is not None:
        same = (actions == SO.inverse_cdf(cdf, u)).mean()
        assert same >= exact_share, same


@pytest.mark.parametrize("N", [129, 4097])
@pytest.mark.parametrize("A", [1, 2, 3, 4, 5, 32, 33, 100, 1024])
def test_sample_categorical_against_float64(ctx, A, N):
    """Each draw of every (seed, counter, env_offset) in STREAMS: key and counter high words, environment ids across 2^32."""
    z = categorical_logits(np.random.default_rng(1000 * A + N), N, A)
    z_dev = _cuda(z)
    for seed, counter, off in STREAMS:
        actions, lp = _sample_categorical(ctx, z_dev, seed, counter, off)
        u = SO.u01(SO.categorical_words(seed, counter, SO.env_ids(off, N))).astype(np.float64)
        # an off-by-one in the walk moves every draw; the band can only excuse draws within cdf_band of a CDF step
        check_categorical_draws(z, actions, lp, u, exact_share=0.99 if A <= 100 else None)


def test_sample_categorical_endpoint_draws(ctx):
    """Draws whose word maps to the largest uniform below 1: the walk must stop at the last action of non-zero probability, never
    fall through to a masked last action (log-prob -inf) or to the last action regardless of its probability."""
    rows = [([0.0, -np.inf], 0), ([0.0, 0.0, -np.inf], 1), ([-np.inf, 0.0], 1)]
    for env_id in SO.TOP_WORD_ENV_IDS:
        assert SO.u01(SO.categorical_words(1, 0, [env_id]))[0] == SO.U01_MAX
        for row, want in rows:
            z = np.array([row], dtype=np.float32)
            actions, lp = _sample_categorical(ctx, _cuda(z), 1, 0, env_id)
            assert actions[0] == want, (env_id, row, actions[0], lp[0])
            assert np.isfinite(lp[0]) and abs(lp[0] - SO.categorical_reference(z)[2][0, want]) <= 2 * EPS, (env_id, row, lp[0])
        # the same draws inside a larger launch and a finite-logit row: the last action can win only by its own mass
        z = np.zeros((3, 4), dtype=np.float32)
        z[:, 3] = -30.0
        actions, lp = _sample_categorical(ctx, _cuda(z), 1, 0, env_id - 1)
        assert actions[1] == 2, actions
        check_categorical_draws(z, actions, lp, SO.u01(SO.categorical_words(1, 0, SO.env_ids(env_id - 1, 3))).astype(np.float64))


# ---------------------------------------------------------------- Gaussian ----------------------------
def gaussian_action_bound(sigma, n, rad, u2, a_ref):
    """Bound on |a - a_ref| for a = fl(mean + expf(log_std) * fl(rad * cs)), rad = sqrtf(-2 logf(u1)), cs = sincosf(fl(2pi_f u2)).

    The fp32 angle fl(2pi_f u2) is off 2pi u2 by u2 (|2pi_f - 2pi| + EPS 2pi_f), up to 5.5e-7 rad, which moves n by at most rad
    times that.  Relative to |n|: logf 1 ulp (halved by the square root) and sqrtf's rounding give 2 EPS, sincosf 2 ulp gives 4 EPS,
    the product's rounding EPS; expf's 2 ulp on sigma 4 EPS; sigma * n and the sum round once each (fused or not) by at most EPS of
    their magnitude.  Each term is rounded up by one part in 2^20 for second-order terms."""
    d_theta = u2 * (abs(TWO_PI_F32 - 2.0 * np.pi) + EPS * TWO_PI_F32)
    return (sigma * rad * d_theta + 12 * EPS * sigma * np.abs(n) + EPS * np.abs(a_ref)) * (1 + 2.0 ** -20)


def gaussian_log_prob_bound(actions, mean, log_std):
    """Bound on the kernel's log-prob against SO.normal_log_prob of its own actions.  Per dimension the kernel computes
    t = -fl(diff^2) / fl(2 sigma sigma) - logf(sigma) - 0.9189385f with diff = fl(a - mean) and sigma = expf(log_std): q = diff^2 /
    (2 sigma^2) is within 13 EPS q (diff 2, square 1, sigma^2 8, product 1, division 1), logf(sigma) within 4 EPS + 2 EPS |log_std|
    of log_std, the constant within 0.92 EPS, and the two subtractions within 2 EPS (q + |log_std| + 0.92).  The running fp32 sum
    over dimensions adds EPS |partial sum| per step, bounded by EPS times the running sums of |t|."""
    d = actions.astype(np.float64) - mean.astype(np.float64)
    ls = log_std.astype(np.float64)
    q = d * d / (2.0 * np.exp(2.0 * ls))
    t = np.abs(q) + np.abs(ls) + 0.5 * np.log(2.0 * np.pi)
    per_dim = EPS * (15.0 * q + 4.0 * np.abs(ls) + 7.0)
    running = EPS * np.cumsum(t, axis=-1).sum(axis=-1)
    return (per_dim.sum(axis=-1) + running) * (1 + 2.0 ** -20)


def check_gaussian_draws(mean, log_std, actions, lp, u1, u2):
    a_ref, n, rad = SO.gaussian_reference(mean, log_std[None, :], u1, u2)
    sigma = np.exp(log_std.astype(np.float64))[None, :]
    err = np.abs(actions.astype(np.float64) - a_ref)
    bound = gaussian_action_bound(sigma, n, rad, u2.astype(np.float64), a_ref)
    assert np.all(err <= bound), (np.argwhere(err > bound)[:8], (err / bound).max())
    lp_ref = SO.normal_log_prob(actions, mean, log_std[None, :])
    lp_err = np.abs(lp.astype(np.float64) - lp_ref)
    lp_bound = gaussian_log_prob_bound(actions, mean, log_std[None, :])
    assert np.all(lp_err <= lp_bound), (np.flatnonzero(lp_err > lp_bound)[:8], (lp_err / lp_bound).max())


@pytest.mark.parametrize("mean_scale", [1.0, 1e3])
@pytest.mark.parametrize("A", [1, 2, 3, 17, 32, 510, 511, 512, 513, 1024])
def test_sample_gaussian_against_float64(ctx, A, mean_scale):
    """Actions and log-probs of every dimension of every draw; per-dimension log_std from -5 to 2."""
    N = 257
    rng = np.random.default_rng(7 * A + int(mean_scale))
    mean = (rng.standard_normal((N, A)) * mean_scale).astype(np.float32)
    log_std = np.linspace(-5.0, 2.0, A).astype(np.float32)
    mean_dev, log_std_dev = _cuda(mean), _cuda(log_std)
    for seed, counter, off in [(SEEDS[0], COUNTERS[0], OFFSETS[0]), (SEEDS[1], COUNTERS[1], OFFSETS[1])]:
        actions, lp = _sample_gaussian(ctx, mean_dev, log_std_dev, seed, counter, off)
        u1, u2 = SO.gaussian_uniforms(seed, counter, SO.env_ids(off, N), A)
        check_gaussian_draws(mean, log_std, actions, lp, u1, u2)


def test_sample_gaussian_noise_does_not_repeat_above_512_dimensions(ctx):
    """Dimension pairs p and p + 256 read distinct Philox counters: the second half of a 1024-dimensional standard normal is not
    a copy of the first."""
    N, A = 64, 1024
    x, _ = _sample_gaussian(ctx, torch.zeros(N, A, device="cuda"), torch.zeros(A, device="cuda"), 3, 11, 0)
    same = x[:, 512:] == x[:, :512]
    assert not same.all(axis=1).any()
    assert same.mean() < 0.01, same.mean()
    assert abs(np.corrcoef(x[:, 512:].ravel(), x[:, :512].ravel())[0, 1]) < 0.05


# ---------------------------------------------------------------- counter base and launch shape ---------
def test_draw_counter_base_adds_to_the_counter(ctx):
    """With the device base at b, a draw at counter c equals a draw at c + b without it and the reference's draw at c + b (the sum
    carries into the counter's high word)."""
    c, b, N = 0xFFFFFFF0, (1 << 33) + 0x20, 300
    rng = np.random.default_rng(11)
    z = categorical_logits(rng, N, 6)
    mean, log_std = rng.standard_normal((N, 5)).astype(np.float32), np.linspace(-1.0, 1.0, 5).astype(np.float32)
    z_dev, mean_dev, log_std_dev = _cuda(z), _cuda(mean), _cuda(log_std)
    base = torch.tensor([b], dtype=torch.int64, device="cuda")
    ctx.set_draw_counter_base(base)
    try:
        based = _sample_categorical(ctx, z_dev, 9, c, 40) + _sample_gaussian(ctx, mean_dev, log_std_dev, 9, c, 40)
    finally:
        ctx.set_draw_counter_base(None)
    plain = _sample_categorical(ctx, z_dev, 9, c + b, 40) + _sample_gaussian(ctx, mean_dev, log_std_dev, 9, c + b, 40)
    for x, y in zip(based, plain):
        assert np.array_equal(x.view(np.uint64 if x.dtype == np.int64 else np.uint32), y.view(np.uint64 if y.dtype == np.int64 else np.uint32))
    assert not np.array_equal(based[0], _sample_categorical(ctx, z_dev, 9, c, 40)[0])      # the base was cleared
    env = SO.env_ids(40, N)
    u = SO.u01(SO.categorical_words(9, SO.draw_counter(c, b), env)).astype(np.float64)
    check_categorical_draws(z, based[0], based[1], u, exact_share=0.99)
    check_gaussian_draws(mean, log_std, based[2], based[3], *SO.gaussian_uniforms(9, SO.draw_counter(c, b), env, 5))


def test_sub_range_launch_equals_the_full_launch(ctx):
    """A launch of rows [lo, hi) with env_offset + lo reproduces those rows of the full launch bit for bit, for both samplers,
    with environment ids across 2^32."""
    N, lo, hi, off = 1000, 37, 803, (1 << 32) - 500
    rng = np.random.default_rng(12)
    z = _cuda(categorical_logits(rng, N, 33))
    mean, log_std = _cuda(rng.standard_normal((N, 17))), _cuda(np.linspace(-3.0, 1.0, 17))
    a, lp = _sample_categorical(ctx, z, 5, 77, off)
    a_sub, lp_sub = _sample_categorical(ctx, z[lo:hi].contiguous(), 5, 77, off + lo)
    assert np.array_equal(a[lo:hi], a_sub) and np.array_equal(lp[lo:hi].view(np.uint32), lp_sub.view(np.uint32))
    x, glp = _sample_gaussian(ctx, mean, log_std, 5, 77, off)
    x_sub, glp_sub = _sample_gaussian(ctx, mean[lo:hi].contiguous(), log_std, 5, 77, off + lo)
    assert np.array_equal(x[lo:hi].view(np.uint32), x_sub.view(np.uint32))
    assert np.array_equal(glp[lo:hi].view(np.uint32), glp_sub.view(np.uint32))
