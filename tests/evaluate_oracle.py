"""NumPy restatement of the evaluation arithmetic (include/dppo.h: dppo_eval_episodes; diamond/evaluation.py).

`EvalBook` carries what the kernel carries across chunks: the running float64 return and length, the episodes recorded and the
count of environments still short of their quota."""
import numpy as np


def quotas(num_episodes: int, num_envs: int) -> np.ndarray:
    """Stable-Baselines3's evaluate_policy split: environment i runs (num_episodes + i) // num_envs episodes."""
    return np.array([(num_episodes + i) // num_envs for i in range(num_envs)], dtype=np.int32)


class EvalBook:
    def __init__(self, quota):
        self.quota = np.asarray(quota, dtype=np.int64)
        n = self.quota.size
        self.slot = np.concatenate([[0], np.cumsum(self.quota)[:-1]]).astype(np.int64)
        self.ep_return, self.ep_len, self.recorded = np.zeros(n), np.zeros(n, np.int64), np.zeros(n, np.int64)
        self.out_returns, self.out_lengths = np.zeros(int(self.quota.sum())), np.zeros(int(self.quota.sum()), np.int64)
        self.remaining = int((self.quota > 0).sum())

    def chunk(self, rewards, terminations, truncations):
        """[T, N] float32 rewards and done masks of one chunk."""
        for t in range(rewards.shape[0]):
            self.step(rewards[t], terminations[t], truncations[t])

    def step(self, rewards, terminations, truncations):
        self.ep_return += np.asarray(rewards, dtype=np.float32).astype(np.float64)
        self.ep_len += 1
        done = (np.asarray(terminations) != 0) | (np.asarray(truncations) != 0)
        for e in np.flatnonzero(done):
            k = self.recorded[e]
            if k < self.quota[e]:
                self.out_returns[self.slot[e] + k] = self.ep_return[e]
                self.out_lengths[self.slot[e] + k] = self.ep_len[e]
                self.recorded[e] += 1
                if self.recorded[e] == self.quota[e]:
                    self.remaining -= 1
            self.ep_return[e], self.ep_len[e] = 0.0, 0
