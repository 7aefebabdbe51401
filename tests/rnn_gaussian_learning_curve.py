"""Learning curve of RecurrentContinuousPPO on device Pendulum-v1, from which the budget and the return bound of
test_rnn_gaussian_gpu.py::test_gaussian_recurrent_agent_learns_device_pendulum are taken.

    python tests/rnn_gaussian_learning_curve.py [--rollouts 400] [--seeds 0 1 2]

Prints, per configuration and seed, the mean episode return over every window of 20 rollouts, the wall time, and the card it ran on
(name, power limit)."""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))


def card():
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def curve(cfg_kw, rollouts, seed, every=20):
    """train()'s loop by hand, recording every rollout's rewards.  Pendulum-v1 episodes all last 200 steps and start together, so the
    mean return of the episodes that finish in a window of rollouts is 200 x the window's mean reward per step."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    N_, T = cfg_kw["num_envs"], cfg_kw["rollout_steps"]
    cfg = RecurrentContinuousPPOConfig(verbose=False, seed=seed, total_steps=N_ * T * rollouts, **cfg_kw)
    agent = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=seed), cfg)
    agent.ticker = None
    agent.current_observations, _ = agent.envs.reset(seed=seed)
    agent.prev_dones = np.zeros(N_, dtype=bool)
    agent.current_hx = torch.zeros(1, N_, cfg.gru_hidden_dim, device=agent.device)
    sums = torch.zeros(rollouts, dtype=torch.float64, device=agent.device)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(rollouts):
        ro = agent.rollout()
        sums[i] = ro.rewards.double().sum()
        agent.learn(ro)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    per_step = (sums / (N_ * T)).cpu().numpy()
    points = [(k + every, 200.0 * float(per_step[k:k + every].mean())) for k in range(0, rollouts - every + 1, every)]
    return dict(points=points, wall_s=wall, last20=points[-1][1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rollouts", type=int, default=400)
    ap.add_argument("--seeds", type=int, nargs="+", default=[0, 1, 2])
    args = ap.parse_args()
    configs = {
        "N64 T32 MB4 gamma0.9 lr1e-3": dict(num_envs=64, rollout_steps=32, num_minibatches=4, gamma=0.9, lr=1e-3),
        "N64 T32 MB4 defaults": dict(num_envs=64, rollout_steps=32, num_minibatches=4),
    }
    print(f"GPU: {card()}", flush=True)
    for name, kw in configs.items():
        for seed in args.seeds:
            res = curve(kw, args.rollouts, seed)
            print(f"{name} seed {seed}: {res['wall_s']:.1f} s, mean return over the last 20 rollouts {res['last20']:.1f}", flush=True)
            print("   " + " ".join(f"{k}:{v:.0f}" for k, v in res["points"]), flush=True)


if __name__ == "__main__":
    main()
