"""Latency of the LSTM networks on the fused kernels (dppo_rnn_desc.cell = 1), on the GPU:
  - learn() with E = 10, MB = 1 (the recurrent defaults) of RecurrentPPO with RecurrentLSTMActorCriticNetwork on the fused engine,
    next to the same network under torch autograd (RecurrentEngine, reached through a subclass), on the same random rollout, at
    Hg = 16 (warp scans), 64 (tiled), 128 and 256 (cluster) and N x T = 32 x 32, 256 x 128 and 4096 x 128;
  - one rollout step of the whole network (base, LSTM step, both heads): dppo_rnn_forward with T = 1 next to the torch module with
    cuDNN's nn.LSTM under inference_mode, at N = 32 and 1024.
Prints the GPU name and power limit first.  Run on the GPU: python tests/lstm_latency.py"""
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
from diamond import RecurrentPPO, RecurrentPPOConfig
from diamond.envs import DeviceVectorEnv
from diamond.recurrent import FusedRecurrentEngine, RecurrentEngine, RecurrentLSTMActorCriticNetwork, RecurrentRollout


class Autograd(RecurrentLSTMActorCriticNetwork):           # a network subclass runs on RecurrentEngine (torch autograd)
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


def rollout(T, N_, D, A, S, dev):
    g = torch.Generator(device=dev).manual_seed(0)
    ro = RecurrentRollout(T, N_, D, S, dev)
    ro.obs.normal_(generator=g); ro.actions.copy_(torch.randint(0, A, (T, N_), device=dev, generator=g))
    ro.rewards.normal_(generator=g); ro.terminations.copy_((torch.rand(T, N_, device=dev, generator=g) < 0.02).float())
    ro.truncations.zero_(); ro.prev_dones.copy_(torch.rand(T, N_, device=dev, generator=g) < 0.02)
    ro.log_probs.fill_(-math.log(A)); ro.values.normal_(generator=g); ro.next_values.normal_(generator=g)
    ro.hx0.zero_(); ro.filled = T
    return ro


def agent(Hg, N_, T, cls):
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, gru_hidden_dim=Hg, verbose=False, seed=1, total_steps=N_ * T * 1000)
    ag = RecurrentPPO(DeviceVectorEnv.factory("CartPole-v1", seed=1), cfg, network_cls=cls)
    assert isinstance(ag.engine, FusedRecurrentEngine if cls is RecurrentLSTMActorCriticNetwork else RecurrentEngine)
    return ag


def learn_ms(Hg, N_, T, cls):
    ag = agent(Hg, N_, T, cls)
    ro = rollout(T, N_, ag.obs_dim, ag.act_dim, ag.state_dim, ag.device)
    np.random.seed(0)
    big = N_ * T >= 4096 * 128
    t = timed(lambda: ag.learn(ro), 2, 3 if big else 10)
    del ag, ro
    torch.cuda.empty_cache()
    return t


def step_ms(Hg, N_):
    """One T = 1 step of the whole network: dppo_rnn_forward against the module with cuDNN nn.LSTM (same parameters)."""
    ag = agent(Hg, N_, 1, RecurrentLSTMActorCriticNetwork)
    eng, dev = ag.engine, ag.device
    net = ag.network
    lstm = torch.nn.LSTM(ag.cfg.network_hidden_dim, Hg).to(dev)
    lstm.load_state_dict({k[len("lstm."):]: v for k, v in net.state_dict().items() if k.startswith("lstm.")})
    obs = torch.randn(1, N_, ag.obs_dim, device=dev)
    pd = torch.zeros(1, N_, dtype=torch.uint8, device=dev)
    hx = torch.randn(N_, 2 * Hg, device=dev) * 0.1
    logits, values, hx_out = torch.empty(1, N_, ag.act_dim, device=dev), torch.empty(1, N_, device=dev), torch.empty(N_, 2 * Hg, device=dev)
    ws = eng._workspace(1, N_, N_, False)
    fused = lambda: ag.ctx.rnn_forward(eng.desc, eng.P, obs, pd, hx, 1, N_, 3, logits, values, hx_out, ws)
    h0, c0 = hx[:, :Hg].unsqueeze(0).contiguous(), hx[:, Hg:].unsqueeze(0).contiguous()

    def cudnn():
        with torch.inference_mode():
            x, _ = lstm(net.base(obs), (h0 * (1 - pd.unsqueeze(-1)), c0 * (1 - pd.unsqueeze(-1))))
            return net.actor_head(x), net.critic_head(x)

    with torch.inference_mode():
        ref_l, _ = cudnn()
    fused()
    torch.cuda.synchronize()
    err = float((logits - ref_l).abs().max())
    return timed(fused, 20, 500), timed(cudnn, 20, 500), err


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}",
          flush=True)
    print(f"{'learn() E=10 MB=1':34s} {'fused':>10s} {'autograd':>10s} {'ratio':>7s}  (ms)")
    for Hg in (16, 64, 128, 256):
        for N_, T in ((32, 32), (256, 128), (4096, 128)):
            lf = learn_ms(Hg, N_, T, RecurrentLSTMActorCriticNetwork)
            la = learn_ms(Hg, N_, T, Autograd)
            print(f"{f'Hg={Hg} N={N_} T={T}':34s} {lf:10.2f} {la:10.2f} {la / lf:6.2f}x", flush=True)
    print(f"{'rollout step (T=1, whole network)':34s} {'fused':>10s} {'cuDNN':>10s} {'ratio':>7s}  (us)   max |logit diff|")
    for Hg in (16, 64, 128, 256):
        for N_ in (32, 1024):
            f, c, err = step_ms(Hg, N_)
            print(f"{f'Hg={Hg} N={N_}':34s} {f * 1e3:10.1f} {c * 1e3:10.1f} {c / f:6.2f}x   {err:.1e}", flush=True)
