"""Latency of RecurrentContinuousPPO on device Pendulum-v1: the default network on the fused engine (FusedRecurrentEngine: device
rollout replayed as a CUDA graph, optimiser steps on dppo_rnn_grad_minibatch) next to the same network under torch autograd
(RecurrentEngine, reached through a subclass of the network; its rollout steps the device environments through the host API).
  - rollout(): T steps of N environments;
  - learn(): E = 10, MB = 1 (the recurrent defaults) on that rollout;
at GRU widths 16 (warp scans), 64 (tiled) and 256 (cluster) and N x T = 32 x 32, 256 x 128 and 4096 x 128.
Prints the GPU name and power limit first.  Run on the GPU: python tests/rnn_gaussian_latency.py"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
from diamond.envs import DeviceVectorEnv
from diamond.recurrent import FusedRecurrentEngine, RecurrentContinuousActorCriticNetwork, RecurrentEngine


class Autograd(RecurrentContinuousActorCriticNetwork):     # a network subclass runs on RecurrentEngine (torch autograd)
    pass


def timed(fn, warm, reps):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps


def measure(Hg, N_, T, cls):
    cfg = RecurrentContinuousPPOConfig(num_envs=N_, rollout_steps=T, gru_hidden_dim=Hg, verbose=False, seed=1, total_steps=N_ * T * 1000)
    ag = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=1), cfg, network_cls=cls)
    assert isinstance(ag.engine, FusedRecurrentEngine if cls is RecurrentContinuousActorCriticNetwork else RecurrentEngine)
    ag.ticker = None
    ag.current_observations, _ = ag.envs.reset(seed=1)
    ag.prev_dones = np.zeros(N_, dtype=bool)
    ag.current_hx = torch.zeros(1, N_, Hg, device=ag.device)
    big = N_ * T >= 4096 * 128
    t_roll = timed(ag.rollout, 3, 3 if big else 10)             # three warm-up rollouts: the fused path replays a graph from the third
    ro = ag.rollout()
    np.random.seed(0)
    t_learn = timed(lambda: ag.learn(ro), 2, 3 if big else 10)
    del ag, ro
    torch.cuda.empty_cache()
    return t_roll, t_learn


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}",
          flush=True)
    print(f"{'':34s} {'rollout fused':>14s} {'autograd':>10s} {'ratio':>7s} {'learn fused':>12s} {'autograd':>10s} {'ratio':>7s}  (ms)")
    for Hg in (16, 64, 256):
        for N_, T in ((32, 32), (256, 128), (4096, 128)):
            rf, lf = measure(Hg, N_, T, RecurrentContinuousActorCriticNetwork)
            ra, la = measure(Hg, N_, T, Autograd)
            print(f"{f'Pendulum-v1 Hg={Hg} N={N_} T={T}':34s} {rf:14.2f} {ra:10.2f} {ra / rf:6.2f}x {lf:12.2f} {la:10.2f} {la / lf:6.2f}x",
                  flush=True)
