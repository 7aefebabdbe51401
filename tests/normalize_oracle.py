"""NumPy float64 restatement of Gymnasium's NormalizeObservation and NormalizeReward wrappers, the checker of the per-environment
normalisation inside diamond.envs.DeviceVectorEnv (csrc/envs.cu; the arithmetic is stated in include/dppo.h).

`RunningMeanStd`, `NormalizeObservation` and `NormalizeReward` follow Gymnasium's code (wrappers/utils.py RunningMeanStd with
update_mean_var_count_from_moments, wrappers/stateful_observation.py and wrappers/stateful_reward.py) with float64 statistics; the
wrappers work around any `diamond.envs.Env` (the host classes).  `PerEnvNormalizer` is the same arithmetic for N environments at
once, fed with the raw stream of a vector environment (observations with a mask of which environments emitted one, rewards with
terminations); every environment's numbers are those of its own wrapper.  No claim is made about bit-agreement with a particular
gymnasium release: the image has no gymnasium, and gymnasium >= 1.0 may keep its RunningMeanStd in the observation space's dtype."""
from __future__ import annotations

import numpy as np


def rms_update(mean, var, count, x):
    """RunningMeanStd.update on a batch of ONE value per statistic (batch mean x, batch variance 0, batch count 1), in NumPy's
    operation order: mean / var arrays (or float64 scalars) and count broadcast against x (float64).  Returns (mean, var, count)."""
    batch_mean, batch_var, batch_count = np.asarray(x, np.float64), 0.0, 1
    delta = batch_mean - mean
    tot_count = count + batch_count
    new_mean = mean + delta * batch_count / tot_count
    m_a = var * count
    m_b = batch_var * batch_count
    M2 = m_a + m_b + np.square(delta) * count * batch_count / tot_count
    return new_mean, M2 / tot_count, tot_count


def normalize_obs(x, mean, var, epsilon, clip=None):
    """float32((x - mean) / sqrt(var + epsilon)), then clipped to [-clip, clip] in float32."""
    y = ((np.asarray(x, np.float32).astype(np.float64) - mean) / np.sqrt(var + epsilon)).astype(np.float32)
    return y if clip is None else np.clip(y, np.float32(-clip), np.float32(clip))


def normalize_reward(r, var, epsilon, clip=None):
    """r / sqrt(var + epsilon) in float64, clipped in float64 (the caller casts to float32 where the reward is stored)."""
    y = np.asarray(r, np.float64) / np.sqrt(var + epsilon)
    return y if clip is None else np.clip(y, -clip, clip)


class RunningMeanStd:
    def __init__(self, shape=()):
        self.mean, self.var, self.count = np.zeros(shape, np.float64), np.ones(shape, np.float64), 1e-4

    def update(self, x):
        self.mean, self.var, self.count = rms_update(self.mean, self.var, self.count, x)


class NormalizeObservation:
    """Gymnasium's NormalizeObservation(env, epsilon) around one host env, + an optional clip (TransformObservation(np.clip))."""

    def __init__(self, env, epsilon=1e-8, clip=None):
        self.env, self.epsilon, self.clip = env, epsilon, clip
        self.obs_rms = RunningMeanStd(env.observation_space.shape)
        self.update_running_mean = True
        self.observation_space = env.observation_space
        self.action_space = env.action_space

    def _obs(self, obs):
        if self.update_running_mean:
            self.obs_rms.update(np.asarray(obs, np.float32))
        return normalize_obs(obs, self.obs_rms.mean, self.obs_rms.var, self.epsilon, self.clip)

    def reset(self, *, seed=None, options=None):
        obs, info = self.env.reset(seed=seed, options=options)
        return self._obs(obs), info

    def close(self):
        self.env.close()

    def step(self, action):
        obs, reward, term, trunc, info = self.env.step(action)
        return self._obs(obs), reward, term, trunc, info


class NormalizeReward:
    """Gymnasium's NormalizeReward(env, gamma, epsilon) around one host env, + an optional clip (TransformReward(np.clip)).
    The accumulator is cut by termination only (not by truncation or reset), as in Gymnasium."""

    def __init__(self, env, gamma=0.99, epsilon=1e-8, clip=None):
        self.env, self.gamma, self.epsilon, self.clip = env, gamma, epsilon, clip
        self.return_rms = RunningMeanStd(())
        self.accumulated_reward = np.array([0.0])
        self.update_running_mean = True
        self.observation_space = env.observation_space
        self.action_space = env.action_space

    def reset(self, *, seed=None, options=None):
        return self.env.reset(seed=seed, options=options)

    def close(self):
        self.env.close()

    def step(self, action):
        obs, reward, term, trunc, info = self.env.step(action)
        self.accumulated_reward = self.accumulated_reward * self.gamma * (1 - term) + float(reward)
        if self.update_running_mean:
            self.return_rms.update(self.accumulated_reward[0])
        return obs, float(normalize_reward(reward, self.return_rms.var, self.epsilon, self.clip)), term, trunc, info


class PerEnvNormalizer:
    """Both wrappers for N environments at once, driven by a vector environment's raw outputs; statistics laid out as
    DeviceVectorEnv's tensors (obs_mean / obs_var [N, D], obs_count [N], return_stats [N, 4] = accumulator, mean, var, count)."""

    def __init__(self, n, d, gamma=0.99, epsilon=1e-8, clip_observation=None, clip_reward=None):
        self.gamma, self.epsilon, self.clip_observation, self.clip_reward = gamma, epsilon, clip_observation, clip_reward
        self.obs_mean, self.obs_var, self.obs_count = np.zeros((n, d)), np.ones((n, d)), np.full(n, 1e-4)
        self.return_stats = np.tile(np.array([0.0, 0.0, 1.0, 1e-4]), (n, 1))
        self.update_running_mean = True

    def observe(self, x, mask=None):
        """Observations x [N, D] (float32) emitted by the environments with mask[e] (None: all); returns the normalised rows."""
        x = np.asarray(x, np.float32)
        m = np.ones(len(x), bool) if mask is None else np.asarray(mask, bool)
        if self.update_running_mean:
            mean, var, count = rms_update(self.obs_mean[m], self.obs_var[m], self.obs_count[m][:, None], x[m].astype(np.float64))
            self.obs_mean[m], self.obs_var[m], self.obs_count[m] = mean, var, count[:, 0]
        return normalize_obs(x, self.obs_mean, self.obs_var, self.epsilon, self.clip_observation)

    def reward(self, r, terminated):
        """One step's float64 rewards [N] and terminations [N]; returns the normalised float64 rewards."""
        st = self.return_stats
        st[:, 0] = st[:, 0] * self.gamma * (1 - np.asarray(terminated, np.int64)) + np.asarray(r, np.float64)
        if self.update_running_mean:
            st[:, 1], st[:, 2], st[:, 3] = rms_update(st[:, 1], st[:, 2], st[:, 3], st[:, 0])
        return normalize_reward(r, st[:, 2], self.epsilon, self.clip_reward)
