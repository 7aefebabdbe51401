"""CPU: the episode split of evaluate() and the NumPy restatement the GPU tests compare dppo_eval_episodes against."""
import numpy as np

from evaluate_oracle import EvalBook, quotas


def test_episode_split_is_stable_baselines3s():
    from diamond.evaluation import episode_quotas
    for num_episodes in (1, 3, 10, 17, 100):
        for num_envs in (1, 2, 4, 7, 8, 64):
            q = episode_quotas(num_episodes, num_envs)
            assert q.dtype == np.int32 and q.sum() == num_episodes
            # evaluate_policy: episode_count_targets = [(n_eval_episodes + i) // n_envs for i in range(n_envs)]
            assert q.tolist() == [(num_episodes + i) // num_envs for i in range(num_envs)]
            assert np.array_equal(q, quotas(num_episodes, num_envs))
    assert episode_quotas(10, 4).tolist() == [2, 2, 3, 3]
    assert episode_quotas(3, 8).tolist() == [0, 0, 0, 0, 0, 1, 1, 1]         # more environments than episodes: quota 0


def test_eval_book_by_hand():
    """Two environments over two chunks.  Env 0 (quota 2) finishes two episodes of 2 steps, the second straddling the chunk
    boundary, then one of 3 steps that is ignored.  Env 1 (quota 1) finishes one episode of 5 steps across the boundary.  Returns
    are float32 rewards summed in float64."""
    book = EvalBook([2, 1])
    r = np.array([[1.0, 0.5], [2.0, 0.25], [0.1, 1.0]], np.float32)
    term = np.array([[0, 0], [1, 0], [0, 0]], np.float32)
    trunc = np.zeros_like(term)
    book.chunk(r, term, trunc)
    assert book.remaining == 2 and book.recorded.tolist() == [1, 0]
    assert book.ep_return[1] == 1.75 and book.ep_len.tolist() == [1, 3]
    r2 = np.array([[3.0, 4.0], [5.0, 8.0], [1.0, 1.0], [1.0, 1.0]], np.float32)
    term2 = np.array([[0, 0], [0, 1], [0, 0], [1, 0]], np.float32)
    trunc2 = np.array([[1, 0], [0, 0], [0, 0], [0, 0]], np.float32)
    book.chunk(r2, term2, trunc2)
    assert book.out_lengths.tolist() == [2, 2, 5]                          # slots: env 0 -> 0, 1; env 1 -> 2
    assert book.out_returns.tolist() == [3.0, np.float64(np.float32(0.1)) + 3.0, 1.75 + 4.0 + 8.0]
    assert book.recorded.tolist() == [2, 1] and book.remaining == 0
    assert book.ep_len.tolist() == [0, 2]                                  # both keep stepping past their quotas


def test_eval_book_ignores_quota_zero_environments():
    book = EvalBook([0, 1])
    assert book.remaining == 1
    book.step(np.ones(2, np.float32), np.ones(2), np.zeros(2))
    assert book.out_lengths.tolist() == [1] and book.remaining == 0 and book.recorded.tolist() == [0, 1]
