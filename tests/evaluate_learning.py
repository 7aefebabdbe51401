"""Greedy evaluation after the training of test_cartpole_learns_on_device, over several seeds: the measurement behind
EVAL_LENGTH_BOUND in tests/test_evaluate_gpu.py.  Prints, per seed, the mean length of the Ticker's last 100 training episodes and
of evaluate(100).

    python tests/evaluate_learning.py [--seeds 1 2 3 4 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "diamond-ppo_b200"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, nargs="+", default=[1, 2, 3, 4, 5])
    args = ap.parse_args()
    from diamond import PPO, PPOConfig
    from diamond.envs import DeviceVectorEnv
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    for seed in args.seeds:
        cfg = PPOConfig(num_envs=64, rollout_steps=128, verbose=False, seed=seed, total_steps=64 * 128 * 40)
        agent = PPO(DeviceVectorEnv.factory("CartPole-v1", seed=seed), cfg)
        agent.train()
        res = agent.evaluate(100)
        print(json.dumps(dict(gpu=gpu, seed=seed, training_window_mean_length=float(np.mean(agent.ticker.recent_lengths)),
                              greedy_mean_length=res["mean_length"], greedy_min_length=int(res["lengths"].min()),
                              greedy_mean_return=res["mean_return"])), flush=True)


if __name__ == "__main__":
    main()
