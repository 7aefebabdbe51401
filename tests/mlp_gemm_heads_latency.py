"""Latency of PPO.learn() / ContinuousPPO.learn() on GEMM heads (shapes the fused head kernel refuses), next to the same network run
under torch autograd (AutogradEngine, reached through a subclass of the network: the only way to run these shapes before GEMM heads
existed).  Default epochs and minibatches (E = 4, MB = 8), one learn() on a synthetic rollout:
  - H = 1024, A = 4 (discrete); H = 512, A = 17 (Gaussian, D = 376: Humanoid-shaped); H = 256, A = 100 (discrete) at N x T = 64 x 128
  - H = 2048, A = 1024 (discrete) at N x T = 16 x 64.
Prints the GPU name and power limit first.  Run on the GPU: python tests/mlp_gemm_heads_latency.py"""
import os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
from diamond import PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig, envs
from diamond.agents import FusedMlpEngine, AutogradEngine, RolloutBuffer
from diamond.networks import ActorCriticNetwork, ContinuousActorCriticNetwork


class AutogradDiscrete(ActorCriticNetwork):             # a network subclass runs on AutogradEngine (torch autograd)
    pass


class AutogradContinuous(ContinuousActorCriticNetwork):
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


def learn_latency(D, H, A, cont, N_, T, reps):
    out = []
    nets = (ContinuousActorCriticNetwork, AutogradContinuous) if cont else (ActorCriticNetwork, AutogradDiscrete)
    rng = np.random.default_rng(0)
    exp = [[rng.standard_normal((N_, D)).astype(np.float32), rng.standard_normal((N_, D)).astype(np.float32),
            rng.standard_normal((N_, A)).astype(np.float32) if cont else rng.integers(0, A, N_), rng.standard_normal(N_),
            rng.random(N_) < 0.02, np.zeros(N_, bool)] for _ in range(T)]
    for cls in nets:
        Agent, Cfg = (ContinuousPPO, ContinuousPPOConfig) if cont else (PPO, PPOConfig)
        cfg = Cfg(num_envs=N_, rollout_steps=T, network_hidden_dim=H, verbose=False, seed=1, total_steps=N_ * T * 1000)
        ag = Agent(lambda: envs.SyntheticEnv(D, A, continuous=cont), cfg, network_cls=cls)
        assert isinstance(ag.engine, FusedMlpEngine if cls in (ActorCriticNetwork, ContinuousActorCriticNetwork) else AutogradEngine)
        if isinstance(ag.engine, FusedMlpEngine):
            assert not ag.engine.fused_heads
        buf = RolloutBuffer.from_lists(ag.ctx, exp, cont, ag.device)
        np.random.seed(0)
        out.append(timed(lambda: ag.learn(buf), 2, reps))
        del ag, buf
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}",
          flush=True)
    print(f"{'':52s} {'fused ms':>10s} {'autograd ms':>12s} {'autograd / fused':>17s}")
    for D, H, A, cont, N_, T, reps in ((8, 1024, 4, False, 64, 128, 5), (376, 512, 17, True, 64, 128, 5), (128, 256, 100, False, 64, 128, 5),
                                       (16, 2048, 1024, False, 16, 64, 3)):
        f, a = learn_latency(D, H, A, cont, N_, T, reps)
        name = f"learn() E=4 MB=8 D={D} H={H} A={A}{' gauss' if cont else ''} N={N_} T={T}"
        print(f"{name:52s} {f:10.2f} {a:12.2f} {a / f:16.2f}x", flush=True)
