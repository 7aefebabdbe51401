"""Learning curves on device Pendulum-v1 with and without per-environment observation / reward normalisation (DeviceVectorEnv's
normalize_observation / normalize_reward, clipped to +-10), from which the setting, budget and bound of
test_env_normalize_gpu.py::test_agent_learns_device_pendulum_with_normalisation are taken.

    python tests/env_normalize_learning_curve.py [--rollouts 600] [--seeds 0 1 2 3 4] [--out curves.json]

Covers ContinuousPPO and RecurrentContinuousPPO at their default hyper-parameters, and RecurrentContinuousPPO at 64 x 32 with 4
minibatches (the setting of tests/rnn_gaussian_learning_curve.py).  Prints the card (name, power limit), then per configuration and
seed the mean RAW episode return over every window of 20 rollouts and the wall time.  Pendulum-v1 episodes all last 200 steps and
start together, so a window's mean return is 200 x its mean raw reward per step."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))

NORM = dict(normalize_observation=True, normalize_reward=True, clip_observation=10.0, clip_reward=10.0)
CONFIGS = {
    "ContinuousPPO defaults": ("ContinuousPPO", {}),
    "RecurrentContinuousPPO defaults": ("RecurrentContinuousPPO", {}),
    "RecurrentContinuousPPO N64 T32 MB4": ("RecurrentContinuousPPO", dict(num_envs=64, rollout_steps=32, num_minibatches=4)),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def curve(agent_name, cfg_kw, norm, rollouts, seed, every=20):
    """train()'s loop by hand, recording every rollout's raw rewards."""
    import diamond
    from diamond.envs import DeviceVectorEnv
    Agent, Cfg = getattr(diamond, agent_name), getattr(diamond, agent_name + "Config")
    cfg = Cfg(verbose=False, seed=seed, **cfg_kw)
    N_, T = cfg.num_envs, cfg.rollout_steps
    cfg.total_steps = N_ * T * rollouts
    env_kw = dict(NORM, gamma=cfg.gamma) if norm else {}
    agent = Agent(DeviceVectorEnv.factory("Pendulum-v1", seed=seed, **env_kw), cfg)
    agent.ticker = None
    agent.current_observations, _ = agent.envs.reset(seed=seed)
    if agent_name.startswith("Recurrent"):
        agent.prev_dones = np.zeros(N_, dtype=bool)
        agent.current_hx = torch.zeros(1, N_, cfg.gru_hidden_dim, device=agent.device)
    sums = torch.zeros(rollouts, dtype=torch.float64, device=agent.device)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(rollouts):
        buf = agent.rollout()
        raw = getattr(buf, "raw_rewards", None)
        sums[i] = (buf.rewards if raw is None else raw).double().sum()
        agent.learn(buf)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    per_step = (sums / (N_ * T)).cpu().numpy()
    points = [(k + every, 200.0 * float(per_step[k:k + every].mean())) for k in range(0, rollouts - every + 1, every)]
    return dict(points=points, wall_s=wall, steps_per_rollout=N_ * T)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rollouts", type=int, default=600)
    ap.add_argument("--seeds", type=int, nargs="+", default=[0, 1, 2, 3, 4])
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    results = dict(card=card(), rollouts=args.rollouts, runs=[])
    print(f"GPU: {results['card']}", flush=True)
    for name in args.configs:
        agent_name, kw = CONFIGS[name]
        for norm in (False, True):
            last = []
            for seed in args.seeds:
                res = curve(agent_name, kw, norm, args.rollouts, seed)
                results["runs"].append(dict(config=name, normalize=norm, seed=seed, **res))
                last.append(res["points"][-1][1])
                print(f"{name} normalize={norm} seed {seed}: {res['wall_s']:.1f} s, {res['steps_per_rollout']} steps/rollout", flush=True)
                print("   " + " ".join(f"{k}:{v:.0f}" for k, v in res["points"]), flush=True)
            print(f"== {name} normalize={norm}: last-20-rollout mean return over seeds {np.mean(last):.0f} "
                  f"(min {np.min(last):.0f}, max {np.max(last):.0f})", flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
