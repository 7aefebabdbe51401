"""Rollout time of device environments with per-environment observation + reward normalisation off and on, alternated in one process:
CartPole-v1 64 x 128 (PPO), Pendulum-v1 64 x 200 (ContinuousPPO) and the synthetic stand-in 4096 x 128 with obs_dim 64 (PPO), every
rollout one CUDA graph replay (after three warm-up rollouts).  Each round times BLOCK rollouts of one arm, then of the other, ending
in a device synchronise; the median over rounds is reported per rollout, with the overhead of normalisation.  Prints the GPU name
and power limit first.  Run on the GPU: python tests/env_normalize_latency.py"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
from diamond import ContinuousPPO, ContinuousPPOConfig, PPO, PPOConfig  # noqa: E402
from diamond.envs import DeviceVectorEnv  # noqa: E402

CASES = [("CartPole-v1", 64, 128, {}), ("Pendulum-v1", 64, 200, {}), ("Synthetic", 4096, 128, dict(obs_dim=64, n_actions=4))]
NORM = dict(normalize_observation=True, normalize_reward=True, clip_observation=10.0, clip_reward=10.0)
ROUNDS, BLOCK = 15, 20


def agent_for(env_id, N_, T, kw, norm):
    cont = env_id == "Pendulum-v1"
    Agent, Cfg = (ContinuousPPO, ContinuousPPOConfig) if cont else (PPO, PPOConfig)
    cfg = Cfg(num_envs=N_, rollout_steps=T, verbose=False, seed=1, total_steps=N_ * T * 10_000)
    agent = Agent(DeviceVectorEnv.factory(env_id, seed=1, **kw, **(NORM if norm else {})), cfg)
    agent.ticker = None
    agent.current_observations, _ = agent.envs.reset(seed=1)
    for _ in range(3):                                   # eager, capture, replay
        agent.rollout()
    assert agent._rollout_graph is not None
    return agent


def block_ms(agent):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(BLOCK):
        agent.rollout()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / BLOCK


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}",
          flush=True)
    for env_id, N_, T, kw in CASES:
        off, on = agent_for(env_id, N_, T, kw, False), agent_for(env_id, N_, T, kw, True)
        t_off, t_on = [], []
        for r in range(ROUNDS):
            pair = [(off, t_off), (on, t_on)] if r % 2 == 0 else [(on, t_on), (off, t_off)]
            for agent, acc in pair:
                acc.append(block_ms(agent))
        m_off, m_on = float(np.median(t_off)), float(np.median(t_on))
        print(f"{env_id:12s} {N_:5d} x {T:3d}: rollout off {m_off:7.3f} ms (min {min(t_off):.3f}, max {max(t_off):.3f}), "
              f"on {m_on:7.3f} ms (min {min(t_on):.3f}, max {max(t_on):.3f}): overhead {m_on - m_off:+.3f} ms "
              f"({100 * (m_on / m_off - 1):+.1f} %), {(m_on - m_off) * 1e3 / T:+.2f} us per step", flush=True)
