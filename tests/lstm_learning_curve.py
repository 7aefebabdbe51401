"""Learning runs of the LSTM agents from which the budgets and bounds of test_lstm_gpu.py's learning tests are taken:
RecurrentPPO with RecurrentLSTMActorCriticNetwork on device CartPole-v1, and RecurrentContinuousPPO with
RecurrentContinuousLSTMActorCriticNetwork on device Pendulum-v1 with observation and reward normalisation.

    python tests/lstm_learning_curve.py [--seeds 0 1 2 3 4]

Each run is the test's own train() call; printed per seed: the mean return of the last 20 finished episodes (what the test
bounds), the wall time, and the card it ran on (name, power limit)."""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def run(task, seed):
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig, RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork, RecurrentLSTMActorCriticNetwork
    from test_lstm_gpu import CARTPOLE_ROLLOUTS, PENDULUM_ROLLOUTS
    N_, T = 64, 32
    if task == "cartpole":
        cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, num_minibatches=4, verbose=False, seed=seed,
                                 total_steps=N_ * T * CARTPOLE_ROLLOUTS)
        agent = RecurrentPPO(DeviceVectorEnv.factory("CartPole-v1", seed=seed), cfg, network_cls=RecurrentLSTMActorCriticNetwork)
    else:
        cfg = RecurrentContinuousPPOConfig(num_envs=N_, rollout_steps=T, num_minibatches=4, verbose=False, seed=seed,
                                           total_steps=N_ * T * PENDULUM_ROLLOUTS)
        env_fn = DeviceVectorEnv.factory("Pendulum-v1", seed=seed, normalize_observation=True, normalize_reward=True)
        agent = RecurrentContinuousPPO(env_fn, cfg, network_cls=RecurrentContinuousLSTMActorCriticNetwork)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    agent.train()
    torch.cuda.synchronize()
    returns = agent.ticker.logs["episode_returns"]
    return float(np.mean(returns[-20:])), time.perf_counter() - t0, float(np.mean(returns[:20]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, nargs="+", default=[0, 1, 2, 3, 4])
    ap.add_argument("--tasks", nargs="+", default=["cartpole", "pendulum"])
    args = ap.parse_args()
    print(f"GPU: {card()}", flush=True)
    for task in args.tasks:
        for seed in args.seeds:
            last, wall, first = run(task, seed)
            print(f"{task} seed {seed}: first 20 episodes {first:.1f}, last 20 episodes {last:.1f}, {wall:.1f} s", flush=True)


if __name__ == "__main__":
    main()
