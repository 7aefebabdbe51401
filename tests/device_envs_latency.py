"""Cost of the device-resident classic-control environments (csrc/envs.cu) for CartPole-v1, Acrobot-v1, MountainCar-v0 and
MountainCarContinuous-v0:
  - the environment-step kernel alone (dppo_env_step with in-kernel resets) at N = 4096 and 65 536: 1000 launches captured in one
    CUDA graph, timed with CUDA events over several replays, so the host's launch rate does not enter the number;
  - one device agent.rollout() at 4096 x 128 after warm-up (from the third rollout it is one CUDA graph replay);
  - for scale, one host rollout (diamond.envs.make + SyncVectorEnv, the reference's path) at N = 64 x 128.
Prints the GPU name and power limit first.  Run on the GPU: python tests/device_envs_latency.py"""
import os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
from diamond import PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig, envs
from diamond.envs import DeviceVectorEnv

IDS = ["CartPole-v1", "Acrobot-v1", "MountainCar-v0", "MountainCarContinuous-v0"]
LAUNCHES = 1000


def kernel_us(env_id, N_):
    env = DeviceVectorEnv(env_id, N_, seed=0)
    g = torch.Generator(device="cuda").manual_seed(0)
    if env.continuous:
        actions = torch.rand(N_, env.act_dim, device="cuda", generator=g) * 2 - 1
    else:
        actions = torch.randint(0, env.act_dim, (N_,), device="cuda", generator=g)
    f = dict(dtype=torch.float32, device="cuda")
    nobs, rew, term, trunc = torch.empty(1, N_, env.obs_dim, **f), torch.empty(1, N_, **f), torch.empty(1, N_, **f), torch.empty(1, N_, **f)

    def steps():
        for _ in range(LAUNCHES):
            env.ctx.env_step(env.desc, env._st, actions, 0, True, None, nobs, None, rew, term, trunc)

    steps()                                              # warm-up (module load), episodes under way
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph):
            steps()
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * LAUNCHES)


def agent_for(env_fn, env_id, N_, T):
    cont = env_id == "MountainCarContinuous-v0"
    Agent, Cfg = (ContinuousPPO, ContinuousPPOConfig) if cont else (PPO, PPOConfig)
    cfg = Cfg(num_envs=N_, rollout_steps=T, verbose=False, seed=1, total_steps=N_ * T * 1000)
    agent = Agent(env_fn, cfg)
    agent.current_observations, _ = agent.envs.reset(seed=1)
    return agent


def rollout_ms(agent, warm, reps):
    for _ in range(warm):
        agent.rollout()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        agent.rollout()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}",
          flush=True)
    for env_id in IDS:
        for N_ in (4096, 65536):
            us = kernel_us(env_id, N_)
            print(f"{env_id:26s} env-step kernel N={N_:6d}: {us:8.2f} us  ({N_ / us:8.1f} M env-steps/s)", flush=True)
    for env_id in IDS:
        ms = rollout_ms(agent_for(DeviceVectorEnv.factory(env_id, seed=1), env_id, 4096, 128), 3, 10)
        print(f"{env_id:26s} device rollout() 4096 x 128: {ms:8.2f} ms  ({4096 * 128 / ms / 1e3:8.1f} M env-steps/s)", flush=True)
        ms = rollout_ms(agent_for(lambda: envs.make(env_id), env_id, 64, 128), 1, 1)
        print(f"{env_id:26s} host rollout() 64 x 128:     {ms:8.2f} ms  ({64 * 128 / ms / 1e3:8.3f} M env-steps/s)", flush=True)
