"""CPU: the float64 restatement of Gymnasium's NormalizeObservation / NormalizeReward (tests/normalize_oracle.py) against hand-computed
updates, the per-environment vector form against one wrapper per sub-environment of a SyncVectorEnv, clipping and freezing, and the
ctypes layout of the extended environment descriptor."""
import ctypes as C
import os
import sys
from fractions import Fraction as F

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import normalize_oracle as NO  # noqa: E402


def _close(x, exact, rtol=1e-14):
    return abs(float(x) - float(exact)) <= rtol * abs(float(exact))


def test_first_two_observation_updates_by_hand():
    """From (mean 0, var 1, count 1e-4), two observations behave as a sample that includes a pseudo-observation of weight 1e-4 at
    mean 0 and variance 1: mean = sum(x) / (n + 1e-4), var = (1e-4 + sum((x - mean)^2) + 1e-4 mean^2) / (n + 1e-4)."""
    c0 = F(1, 10000)
    xs = [np.float32(2.0), np.float32(-0.75)]
    rms = NO.RunningMeanStd((1,))
    for n in (1, 2):
        rms.update(np.array([xs[n - 1]], np.float32))
        x = [F(float(v)) for v in xs[:n]]
        mean = sum(x) / (n + c0)
        var = (c0 + sum((v - mean) ** 2 for v in x) + c0 * mean ** 2) / (n + c0)
        assert _close(rms.mean[0], mean) and _close(rms.var[0], var), (n, rms.mean, rms.var)
        assert rms.count == float(n + c0) or _close(rms.count, n + c0)
    # after the first update: mean = 2 / 1.0001, var = (1e-4 + 4e-4 / 1.0001) / 1.0001
    m1, v1, c1 = NO.rms_update(np.zeros(1), np.ones(1), 1e-4, np.array([2.0]))
    assert m1[0] == 2.0 / 1.0001 and v1[0] == (1e-4 + 4.0 * 1e-4 / 1.0001) / 1.0001 and c1 == 1.0001
    y = NO.normalize_obs(np.array([2.0], np.float32), m1, v1, 1e-8)
    assert y.dtype == np.float32 and y[0] == np.float32((2.0 - m1[0]) / np.sqrt(v1[0] + 1e-8))


def test_reward_steps_with_a_termination_by_hand():
    """acc = acc * gamma * (1 - terminated) + r: a termination cuts what came before the terminal reward, a truncation cuts nothing."""
    g, c0 = 0.9, F(1, 10000)
    nz = NO.PerEnvNormalizer(1, 1, gamma=g)
    steps = [(1.0, False), (2.0, True), (3.0, False)]       # the third step may follow a truncation: nothing is cut
    accs = [1.0, 2.0, 2.0 * 0.9 + 3.0]
    for k, ((r, term), acc) in enumerate(zip(steps, accs)):
        out = nz.reward(np.array([r]), np.array([term]))
        assert nz.return_stats[0, 0] == acc
        a = [F(v) for v in accs[:k + 1]]
        n = k + 1
        mean = sum(a) / (n + c0)
        var = (c0 + sum((v - mean) ** 2 for v in a) + c0 * mean ** 2) / (n + c0)
        assert _close(nz.return_stats[0, 1], mean) and _close(nz.return_stats[0, 2], var)
        assert out[0] == r / np.sqrt(nz.return_stats[0, 2] + 1e-8)
    w = NO.NormalizeReward(_Scripted([(1.0, False), (2.0, True), (3.0, False)]), gamma=g)
    got = [w.step(0)[1] for _ in range(3)]
    np.testing.assert_array_equal(got, [float(nz2) for nz2 in _replay_rewards(steps, g)])


def _replay_rewards(steps, g):
    nz = NO.PerEnvNormalizer(1, 1, gamma=g)
    return [nz.reward(np.array([r]), np.array([t]))[0] for r, t in steps]


class _Scripted:
    """Host env that replays (reward, terminated) pairs with a 1-feature observation."""

    def __init__(self, script):
        from diamond.envs import Box, Discrete
        self.script, self.k = script, 0
        self.observation_space, self.action_space = Box(-np.inf, np.inf, (1,)), Discrete(2)

    def reset(self, *, seed=None, options=None):
        return np.zeros(1, np.float32), {}

    def step(self, action):
        r, t = self.script[self.k]
        self.k += 1
        return np.full(1, self.k, np.float32), r, t, False, {}


def _wrapped(env_id, clip_obs, clip_rew, gamma):
    from diamond import envs

    def fn():
        return NO.NormalizeReward(NO.NormalizeObservation(envs.make(env_id), clip=clip_obs), gamma=gamma, clip=clip_rew)
    return fn


@pytest.mark.parametrize("env_id,clip_obs,clip_rew", [("CartPole-v1", None, None), ("Pendulum-v1", 2.0, 0.5), ("Acrobot-v1", None, 1.0),
                                                      ("MountainCarContinuous-v0", 1.5, None)])
def test_per_env_oracle_equals_one_wrapper_per_sub_env(env_id, clip_obs, clip_rew):
    """The vector oracle fed with a plain SyncVectorEnv's raw stream equals a SyncVectorEnv of wrapped sub-environments, bit for bit:
    observations (final and post-reset), rewards and every environment's statistics."""
    from diamond import envs
    n, steps, gamma = 6, 400, 0.97
    raw = envs.SyncVectorEnv([lambda: envs.make(env_id) for _ in range(n)])
    wrapped = envs.SyncVectorEnv([_wrapped(env_id, clip_obs, clip_rew, gamma) for _ in range(n)])
    D = raw.single_observation_space.shape[0]
    nz = NO.PerEnvNormalizer(n, D, gamma=gamma, clip_observation=clip_obs, clip_reward=clip_rew)
    o_raw, _ = raw.reset(seed=5)
    o_w, _ = wrapped.reset(seed=5)
    np.testing.assert_array_equal(nz.observe(o_raw), o_w)
    rng = np.random.default_rng(0)
    cont = isinstance(raw.single_action_space, envs.Box)
    done_any = 0
    for t in range(steps):
        a = rng.uniform(-2, 2, (n, 1)).astype(np.float32) if cont else rng.integers(0, raw.single_action_space.n, n)
        if env_id == "MountainCarContinuous-v0" and t % 50 == 0:          # a few terminations of the continuous car
            for sub in raw.envs + [w.env.env for w in wrapped.envs]:
                sub.state = np.array([0.449, 0.05], np.float32)
        o1, r1, te1, tr1, _ = raw.step(a)
        o2, r2, te2, tr2, _ = wrapped.step(a)
        np.testing.assert_array_equal(te1, te2)
        np.testing.assert_array_equal(nz.observe(o1), o2)
        np.testing.assert_array_equal(nz.reward(r1, te1), r2)
        dones = te1 | tr1
        if t == 150:                                                   # a reset the env did not ask for: the accumulator runs on
            dones = dones | (np.arange(n) == 0)
        if dones.any():
            done_any += 1
            o1, _ = raw.reset(options={"reset_mask": dones})
            o2, _ = wrapped.reset(options={"reset_mask": dones})
            np.testing.assert_array_equal(nz.observe(o1, dones)[dones], o2[dones])
    assert done_any > 0
    for i, w in enumerate(wrapped.envs):
        np.testing.assert_array_equal(nz.obs_mean[i], w.env.obs_rms.mean)
        np.testing.assert_array_equal(nz.obs_var[i], w.env.obs_rms.var)
        assert nz.obs_count[i] == w.env.obs_rms.count
        assert nz.return_stats[i, 0] == w.accumulated_reward[0]
        assert (nz.return_stats[i, 1], nz.return_stats[i, 2], nz.return_stats[i, 3]) == \
            (w.return_rms.mean, w.return_rms.var, w.return_rms.count)


def test_clipping():
    rng = np.random.default_rng(1)
    a, b = NO.PerEnvNormalizer(8, 5, clip_observation=1.25, clip_reward=0.3), NO.PerEnvNormalizer(8, 5)
    for _ in range(20):                                                # then an outlier of 50 standard deviations
        x = rng.standard_normal((8, 5)).astype(np.float32)
        np.testing.assert_array_equal(a.observe(x), np.clip(b.observe(x), np.float32(-1.25), np.float32(1.25)))
        r = rng.standard_normal(8) * 0.01
        np.testing.assert_array_equal(a.reward(r, np.zeros(8, bool)), np.clip(b.reward(r, np.zeros(8, bool)), -0.3, 0.3))
    x = (rng.standard_normal((8, 5)) * 50).astype(np.float32)
    ya, yb = a.observe(x), b.observe(x)
    assert np.abs(ya).max() == np.float32(1.25) and np.abs(yb).max() > 1.25
    np.testing.assert_array_equal(ya, np.clip(yb, np.float32(-1.25), np.float32(1.25)))
    r = rng.standard_normal(8) * 100
    ra, rb = a.reward(r, np.zeros(8, bool)), b.reward(r, np.zeros(8, bool))
    assert np.abs(ra).max() == 0.3 and np.abs(rb).max() > 0.3
    np.testing.assert_array_equal(ra, np.clip(rb, -0.3, 0.3))
    np.testing.assert_array_equal(a.obs_mean, b.obs_mean)             # clipping acts on the output only
    np.testing.assert_array_equal(a.return_stats, b.return_stats)


def test_freezing_keeps_the_statistics_and_runs_the_accumulator():
    rng = np.random.default_rng(2)
    nz = NO.PerEnvNormalizer(4, 3, gamma=0.5)
    for _ in range(5):
        nz.observe(rng.standard_normal((4, 3)))
        nz.reward(rng.standard_normal(4), np.zeros(4, bool))
    mean, var, count, rs = nz.obs_mean.copy(), nz.obs_var.copy(), nz.obs_count.copy(), nz.return_stats.copy()
    nz.update_running_mean = False
    x, r = rng.standard_normal((4, 3)).astype(np.float32), rng.standard_normal(4)
    y, out = nz.observe(x), nz.reward(r, np.array([True, False, False, False]))
    np.testing.assert_array_equal(nz.obs_mean, mean)
    np.testing.assert_array_equal(nz.obs_var, var)
    np.testing.assert_array_equal(nz.obs_count, count)
    np.testing.assert_array_equal(nz.return_stats[:, 1:], rs[:, 1:])
    np.testing.assert_array_equal(nz.return_stats[:, 0], rs[:, 0] * 0.5 * np.array([0, 1, 1, 1]) + r)
    np.testing.assert_array_equal(y, NO.normalize_obs(x, mean, var, 1e-8))
    np.testing.assert_array_equal(out, r / np.sqrt(rs[:, 2] + 1e-8))
    w = NO.NormalizeObservation(_Scripted([(0.0, False)] * 3))
    w.step(0)
    w.update_running_mean = False
    before = (w.obs_rms.mean.copy(), w.obs_rms.var.copy(), w.obs_rms.count)
    w.step(0)
    assert (w.obs_rms.mean, w.obs_rms.var, w.obs_rms.count) == before


def test_env_descriptor_layout_and_zero_default():
    """dppo_env_desc grew at its end: today's positional EnvDesc(...) leaves normalisation off, and the fields sit where the C
    struct puts them (natural alignment)."""
    from diamond import _native as N
    d = N.EnvDesc(0, 8, 4, 2, 1, 0, 0.0, 0.0)
    assert d.normalize == 0 and d.gamma == 0.0 and d.epsilon == 0.0 and d.clip_observation == 0.0 and d.clip_reward == 0.0
    assert N.EnvDesc.normalize.offset == 40 and N.EnvDesc.gamma.offset == 48 and N.EnvDesc.clip_reward.offset == 72
    assert C.sizeof(N.EnvDesc) == 80
    assert [f for f, _ in N.EnvState._fields_][5:] == ["obs_mean", "obs_var", "obs_count", "ret_stats", "update"]
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "dppo.h")).read()
    desc = hdr[hdr.index("typedef struct dppo_env_desc"):hdr.index("} dppo_env_desc;")]
    for name in ("normalize", "gamma", "epsilon", "clip_observation", "clip_reward"):
        assert name in desc
    assert N.ENV_NORMALIZE_OBS == 1 and N.ENV_NORMALIZE_REWARD == 2
    assert "#define DPPO_ENV_NORMALIZE_OBS 1" in hdr and "#define DPPO_ENV_NORMALIZE_REWARD 2" in hdr
