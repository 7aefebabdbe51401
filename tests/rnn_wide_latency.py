"""Latency of RecurrentPPO's default network at GRU widths 128 (tiled scans, the reference point), 256 and 512 (cluster scans),
next to the same network run under torch autograd (RecurrentEngine, reached through a subclass of the network: the only way to
run these widths before the cluster scans existed).
  - one rollout step: dppo_rnn_forward at T = 1 (FusedRecurrentEngine.forward) against the module's get_logits_values_and_hx under
    inference_mode, N = 32 and 1024;
  - RecurrentPPO.learn() at the default shape (N = 32, T = 32, E = 10, MB = 1) and at N = 256 / 4096 with T = 128.
Prints the GPU name and power limit first.  Run on the GPU: python tests/rnn_wide_latency.py"""
import os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
from diamond import RecurrentPPO, RecurrentPPOConfig, envs
from diamond.recurrent import RecurrentActorCriticNetwork, RecurrentRollout, FusedRecurrentEngine, RecurrentEngine

D, A = 4, 2                                             # CartPole-sized observations and actions


class Autograd(RecurrentActorCriticNetwork):            # a network subclass runs on RecurrentEngine (torch autograd)
    pass


def agent(Hg, N_, T, cls):
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, gru_hidden_dim=Hg, verbose=False, seed=1, total_steps=N_ * T * 1000)
    ag = RecurrentPPO(lambda: envs.SyntheticEnv(D, A), cfg, network_cls=cls)
    assert isinstance(ag.engine, FusedRecurrentEngine if cls is RecurrentActorCriticNetwork else RecurrentEngine)
    return ag


def timed(fn, warm, reps):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps


def step_latency(Hg, N_):
    out = []
    for cls in (RecurrentActorCriticNetwork, Autograd):
        ag = agent(Hg, N_, 1, cls)
        g = torch.Generator(device="cuda").manual_seed(0)
        obs = torch.randn(1, N_, D, device="cuda", generator=g)
        hx = torch.randn(1, N_, Hg, device="cuda", generator=g)
        pd = torch.rand(1, N_, device="cuda", generator=g) < 0.05
        if cls is RecurrentActorCriticNetwork:
            fn = lambda: ag.engine.forward(obs, hx, pd, heads=3)
        else:
            def fn():
                with torch.inference_mode():
                    ag.network.get_logits_values_and_hx(obs, hx, pd)
        out.append(timed(fn, 20, 200))
    return out


def learn_latency(Hg, N_, T):
    out = []
    for cls in (RecurrentActorCriticNetwork, Autograd):
        ag = agent(Hg, N_, T, cls)
        g = torch.Generator(device="cuda").manual_seed(Hg)
        ro = RecurrentRollout(T, N_, D, Hg, ag.device)
        ro.obs.normal_(generator=g); ro.actions.random_(0, A, generator=g); ro.rewards.normal_(generator=g)
        ro.terminations.copy_((torch.rand(T, N_, device="cuda", generator=g) < 0.02).float()); ro.truncations.zero_()
        ro.prev_dones.copy_(torch.rand(T, N_, device="cuda", generator=g) < 0.02)
        ro.log_probs.fill_(-float(np.log(A))); ro.values.normal_(generator=g); ro.next_values.normal_(generator=g)
        ro.hx0.normal_(generator=g); ro.filled = T
        np.random.seed(0)
        reps = 3 if N_ * T * Hg >= 4096 * 128 * 256 else 10
        out.append(timed(lambda: ag.learn(ro), 2, reps))
        del ag, ro
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}",
          flush=True)
    print(f"{'':44s} {'fused ms':>10s} {'autograd ms':>12s} {'autograd / fused':>17s}")
    for Hg in (128, 256, 512):
        for N_ in (32, 1024):
            f, a = step_latency(Hg, N_)
            print(f"{f'rollout step T=1 Hg={Hg} N={N_}':44s} {f:10.3f} {a:12.3f} {a / f:16.2f}x", flush=True)
    for Hg in (128, 256, 512):
        for N_, T in ((32, 32), (256, 128), (4096, 128)):
            f, a = learn_latency(Hg, N_, T)
            print(f"{f'learn() E=10 MB=1 Hg={Hg} N={N_} T={T}':44s} {f:10.2f} {a:12.2f} {a / f:16.2f}x", flush=True)
