"""Cost of evaluate(100) on device CartPole-v1 and Pendulum-v1 at N = 64 and 1024 environments, for the default MLP and GRU agents,
against a user's host loop through the torch module (module forward under inference_mode, argmax / means, DeviceVectorEnv.step
with host arrays, masked resets).  Both loops play the same greedy episodes on the same environments.

    python tests/evaluate_latency.py [--out evaluate_latency.json] [--repeats 3]
"""
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
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from evaluate_oracle import EvalBook, quotas  # noqa: E402


def torch_module_loop(agent, env_fn, n, episodes, seed):
    """What a user writes without evaluate(): the torch module step by step, host arrays through the environment API."""
    envs = env_fn(n)
    book = EvalBook(quotas(episodes, n))
    obs, _ = envs.reset(seed=seed)
    recurrent = agent.__class__.__name__.startswith("Recurrent")
    net, dev = agent.network, agent.device
    hx = torch.zeros(1, n, agent.cfg.gru_hidden_dim, device=dev) if recurrent else None
    prev = np.zeros(n, dtype=bool)
    while book.remaining > 0:
        x = torch.as_tensor(obs, device=dev)
        with torch.inference_mode():
            if recurrent:
                pd = torch.as_tensor(prev, device=dev)[None]
                if agent._continuous:
                    head, _, _, hx = net.get_means_log_stds_values_and_hx(x[None], hx, pd)
                else:
                    head, _, hx = net.get_logits_values_and_hx(x[None], hx, pd)
                head = head[0]
            elif agent._continuous:
                head, _, _ = net.get_means_log_stds_and_values(x)
            else:
                head, _ = net.get_logits_and_values(x)
        actions = head if agent._continuous else torch.argmax(head, -1)
        nobs, rew, term, trunc, _ = envs.step(actions.cpu().numpy())
        book.step(rew, term, trunc)
        dones = term | trunc
        obs = envs.reset(options={"reset_mask": dones})[0] if dones.any() else nobs
        prev = dones
    return book.out_lengths


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    from diamond import (PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig, RecurrentPPO, RecurrentPPOConfig, RecurrentContinuousPPO,
                         RecurrentContinuousPPOConfig)
    from diamond.envs import DeviceVectorEnv
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    rows = []
    for env_id, agents in (("CartPole-v1", ((PPO, PPOConfig, "mlp"), (RecurrentPPO, RecurrentPPOConfig, "gru"))),
                           ("Pendulum-v1", ((ContinuousPPO, ContinuousPPOConfig, "mlp"), (RecurrentContinuousPPO, RecurrentContinuousPPOConfig, "gru")))):
        for Agent, Cfg, net in agents:
            for n in (64, 1024):
                env_fn = DeviceVectorEnv.factory(env_id, seed=1)
                agent = Agent(env_fn, Cfg(num_envs=n, rollout_steps=32, verbose=False, seed=1))
                agent.evaluate(100, seed=5)                           # warm-up: modules, workspaces, graph capture
                times = []
                for _ in range(args.repeats):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res = agent.evaluate(100, seed=5)
                    times.append(time.perf_counter() - t0)
                torch_module_loop(agent, env_fn, n, 100, 5)
                host_times = []
                for _ in range(args.repeats):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    lengths = torch_module_loop(agent, env_fn, n, 100, 5)
                    torch.cuda.synchronize()
                    host_times.append(time.perf_counter() - t0)
                row = dict(env=env_id, net=net, N=n, evaluate_ms=1e3 * min(times), torch_loop_ms=1e3 * min(host_times),
                           speedup=min(host_times) / min(times), mean_length=res["mean_length"],
                           same_lengths=bool(np.array_equal(np.sort(lengths), np.sort(res["lengths"]))))
                print(json.dumps(row), flush=True)
                rows.append(row)
    out = dict(gpu=gpu, rows=rows)
    print(json.dumps(dict(gpu=gpu)))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
