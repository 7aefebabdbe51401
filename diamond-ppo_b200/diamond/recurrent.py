"""RecurrentPPO (reference: diamond/recurrent_ppo.py) on the libdppo kernels.

Kept from the reference: `RecurrentPPO(env_fn, cfg, network_cls)`, `RecurrentPPOConfig`, `GRUCore`,
`RecurrentActorCriticNetwork` with `get_values(obs[T,B,D], hx, dones)` /
`get_logits_values_and_hx(obs, hx, dones) -> (logits, values, hx)` (recurrent_ppo.py:127-149), the attributes
`current_observations / current_hx / prev_dones` and `rollout() / calculate_advantage() / learn() / train()`.

What runs where.  Default network class (`RecurrentActorCriticNetwork`): everything on libdppo kernels -- the base layer, the
input projection of all T steps, the GRU recurrence with done-masked hidden resets (forward scan), the heads + PPO loss,
back-propagation through all T steps (backward scan), weight gradients, clip and Adam (`FusedRecurrentEngine`,
csrc/rnn.cu: `dppo_rnn_forward`, `dppo_rnn_grad_minibatch`); parameters are views of one flat buffer.
Custom `network_cls`: the user module runs under torch autograd (its GRU time loop restructured as ONE input-projection
GEMM over all T steps followed by T hidden-state steps, instead of T one-step `nn.GRU` calls) and only GAE + returns,
advantage normalisation, the bit-exact minibatch permutation, the PPO loss forward/backward, gradient clipping and Adam run
on the libdppo kernels (`RecurrentEngine`).  The reference's `hx or zeros` / `dones or zeros` lines (recurrent_ppo.py:78-79) raise on
every call; the intended `is None` semantics are implemented (SURVEY.md §0.4).

Beyond the reference: `RecurrentContinuousPPO` / `RecurrentContinuousActorCriticNetwork`, the same agent with a Gaussian policy for
Box action spaces (the heads of continuous_ppo.py on the GRU trunk).  It runs the same code, selected by the class attribute
`_continuous` as in agents.py, and the same kernels (the Gaussian instantiation of the head kernel in dppo_rnn_grad_minibatch).
"""
from __future__ import annotations

import time
from math import sqrt
from typing import Any, Callable

import numpy as np
import torch
import torch.nn as nn

from . import _native as N
try:                                    # the real package when present, else the in-repo shim (same rule as agents.py)
    import gymnasium as gym             # noqa: F401
except ImportError:                     # pragma: no cover - the GPU image has no gymnasium
    from . import envs as gym
from .agents import _Dist, _EngineBase, _PermWorker, _PPOBase, _require_cuda
from .config import RecurrentContinuousPPOConfig, RecurrentPPOConfig
from .evaluation import PolicyEvaluation, as_device_obs, select_actions, shared_log_std
from .networks import _obs_dim, network_parameter_init_
from .utils import Checkpointer, Logger, Ticker, Timer


class GRUCore(nn.GRU):
    """GRU for RL with per-timestep hidden state resets (recurrent_ppo.py:41-91).  Parameters are nn.GRU's
    (`weight_ih_l0 [3Hg, H]`, `weight_hh_l0 [3Hg, Hg]`, `bias_ih_l0`, `bias_hh_l0`; gate order r, z, n), so state dicts are
    interchangeable with the reference."""

    def __init__(self, input_dim: int, hidden_dim: int) -> None:
        super().__init__(input_dim, hidden_dim)

    def forward(self, x: torch.Tensor, hx: torch.Tensor | None, dones: torch.Tensor | None):
        T, B = x.shape[:2]
        Hg = self.hidden_size
        h = torch.zeros(B, Hg, dtype=x.dtype, device=x.device) if hx is None else hx.reshape(B, Hg)
        # all T input projections in one GEMM; only the hidden-to-hidden product is sequential
        gi = torch.addmm(self.bias_ih_l0, x.reshape(T * B, -1), self.weight_ih_l0.t()).view(T, B, 3 * Hg)
        keep = None if dones is None else (~dones.to(torch.bool)).to(x.dtype).unsqueeze(-1)      # [T, B, 1]
        outs = []
        for t in range(T):
            if keep is not None:
                h = h * keep[t]                                   # reset hidden state at the start of new episodes (:84)
            gh = torch.addmm(self.bias_hh_l0, h, self.weight_hh_l0.t())
            i_r, i_z, i_n = gi[t].chunk(3, dim=-1)
            h_r, h_z, h_n = gh.chunk(3, dim=-1)
            r = torch.sigmoid(i_r + h_r)
            z = torch.sigmoid(i_z + h_z)
            n = torch.tanh(i_n + r * h_n)
            h = (1.0 - z) * n + z * h
            outs.append(h)
        return torch.stack(outs, dim=0), h.unsqueeze(0)


class RecurrentActorCriticNetwork(nn.Module):
    """Linear-Tanh -> GRU -> actor / critic heads (recurrent_ppo.py:94-149)."""

    def __init__(self, observation_space, action_space, cfg: RecurrentPPOConfig) -> None:
        super().__init__()
        assert hasattr(action_space, "n"), "Only Discrete action spaces are supported."
        d, h, hg = _obs_dim(observation_space), int(cfg.network_hidden_dim), int(cfg.gru_hidden_dim)
        self.base = nn.Sequential(nn.Linear(d, h), nn.Tanh())
        self.gru = GRUCore(h, hg)
        self.actor_head = nn.Sequential(nn.Linear(hg, h), nn.Tanh(), nn.Linear(h, int(action_space.n)))
        self.actor_out_layer = self.actor_head[-1]
        self.critic_head = nn.Sequential(nn.Linear(hg, h), nn.Tanh(), nn.Linear(h, 1))

    def get_values(self, observations, hx, dones) -> torch.Tensor:
        x, _ = self.gru.forward(self.base(observations), hx, dones)
        return self.critic_head(x).squeeze(-1)

    def get_logits_values_and_hx(self, observations, hx, dones):
        x, hx = self.gru.forward(self.base(observations), hx, dones)
        return self.actor_head(x), self.critic_head(x).squeeze(-1), hx


class RecurrentContinuousActorCriticNetwork(nn.Module):
    """Linear-Tanh -> GRU -> Gaussian actor (mean head + state-independent log-std parameter (1, A), as in
    ContinuousActorCriticNetwork) / critic head."""

    def __init__(self, observation_space, action_space, cfg: RecurrentContinuousPPOConfig) -> None:
        super().__init__()
        assert hasattr(action_space, "shape") and not hasattr(action_space, "n"), "Only Box action spaces are supported."
        d, h, hg = _obs_dim(observation_space), int(cfg.network_hidden_dim), int(cfg.gru_hidden_dim)
        a = int(np.prod(action_space.shape))
        self.base = nn.Sequential(nn.Linear(d, h), nn.Tanh())
        self.gru = GRUCore(h, hg)
        self.actor_mean_head = nn.Sequential(nn.Linear(hg, h), nn.Tanh(), nn.Linear(h, a))
        self.actor_log_std = nn.Parameter(torch.zeros(1, a))
        self.critic_head = nn.Sequential(nn.Linear(hg, h), nn.Tanh(), nn.Linear(h, 1))

    def get_values(self, observations, hx, dones) -> torch.Tensor:
        x, _ = self.gru.forward(self.base(observations), hx, dones)
        return self.critic_head(x).squeeze(-1)

    def get_means_log_stds_values_and_hx(self, observations, hx, dones):
        """(mean [T,B,A], log_std broadcast to [T,B,A], values [T,B], hx [1,B,Hg])."""
        x, hx = self.gru.forward(self.base(observations), hx, dones)
        mean = self.actor_mean_head(x)
        return mean, torch.broadcast_to(self.actor_log_std, mean.shape), self.critic_head(x).squeeze(-1), hx


class RecurrentRollout:
    """Device-resident rollout of the recurrent agent; iterating yields the reference's 10-item step records
    (recurrent_ppo.py:234-245).  Actions: int64 [T, N], or f32 [T, N, act_dim] when act_dim is given (Gaussian policy)."""

    def __init__(self, T, N_, D, Hg, device, act_dim=None):
        f = dict(dtype=torch.float32, device=device)
        self.T, self.N = T, N_
        self.obs = torch.empty(T, N_, D, **f)
        self.actions = torch.empty(T, N_, dtype=torch.int64, device=device) if act_dim is None else torch.empty(T, N_, act_dim, **f)
        self.rewards, self.terminations, self.truncations = (torch.empty(T, N_, **f) for _ in range(3))
        self.prev_dones = torch.empty(T, N_, dtype=torch.bool, device=device)
        self.log_probs, self.values, self.next_values = (torch.empty(T, N_, **f) for _ in range(3))
        self.hx0 = torch.zeros(1, N_, Hg, **f)
        self.filled = 0

    @staticmethod
    def from_lists(experience, device, continuous=False) -> "RecurrentRollout":
        cols = list(zip(*experience))
        dev_t = lambda x, dt: torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x).to(device=device, dtype=dt)
        obs = torch.stack([dev_t(o, torch.float32) for o in cols[0]])
        T, N_, D = obs.shape
        hx0 = dev_t(cols[9][0], torch.float32).clone()                  # recurrent_ppo.py:313
        actions = torch.stack([dev_t(a, torch.float32 if continuous else torch.int64) for a in cols[1]])
        r = RecurrentRollout(T, N_, D, hx0.shape[-1], device, actions.reshape(T, N_, -1).shape[-1] if continuous else None)
        r.obs.copy_(obs)
        r.actions.copy_(actions.reshape(r.actions.shape))
        r.rewards.copy_(dev_t(np.asarray([np.asarray(x) for x in cols[2]]), torch.float32))       # f64 -> f32 (:306)
        r.terminations.copy_(dev_t(np.asarray([np.asarray(x) for x in cols[3]]), torch.float32))
        r.truncations.copy_(dev_t(np.asarray([np.asarray(x) for x in cols[4]]), torch.float32))
        r.prev_dones.copy_(torch.stack([dev_t(p, torch.bool) for p in cols[5]]))
        r.log_probs.copy_(torch.stack([dev_t(x, torch.float32) for x in cols[6]]))
        r.values.copy_(torch.stack([dev_t(x, torch.float32) for x in cols[7]]))
        r.next_values.copy_(torch.stack([dev_t(x, torch.float32) for x in cols[8]]))
        r.hx0.copy_(hx0.reshape(r.hx0.shape))
        r.filled = T
        return r

    def __len__(self):
        return self.filled

    def __iter__(self):
        for t in range(self.filled):
            yield [self.obs[t], self.actions[t], self.rewards[t].cpu().numpy(), self.terminations[t].bool().cpu().numpy(),
                   self.truncations[t].bool().cpu().numpy(), self.prev_dones[t], self.log_probs[t], self.values[t],
                   self.next_values[t], self.hx0]


class RecurrentEngine(_EngineBase):
    """learn() of the recurrent agent: sequence forward/backward under autograd, everything else on libdppo kernels."""

    def __init__(self, ctx, network, cfg, device, dist: _Dist | None = None, continuous=False):
        self.ctx, self.cfg, self.device, self.continuous = ctx, cfg, device, continuous
        self.dist = dist if dist is not None else _Dist(None, False)
        self.network = network
        offsets, o = {}, 0
        for name, p in network.named_parameters():
            offsets[name] = (o, tuple(p.shape))
            o += (p.numel() + 3) // 4 * 4
        self._adopt(network, offsets, max(o, 4))
        self.last_losses = None
        self.draws = 0
        self.seed = self.dist.shared_seed(cfg.seed if cfg.seed is not None else (None if self.dist.enabled else int(np.random.randint(0, 2 ** 31 - 1))), device)
        self.env_offset = self.dist.rank * cfg.num_envs              # global id of this shard's first environment (sampling keys)

    def learn(self, ro: RecurrentRollout):
        cfg, ctx, net, dev, dist = self.cfg, self.ctx, self.network, self.device, self.dist
        T, N_ = ro.T, ro.N
        E, MB = cfg.num_epochs, cfg.num_minibatches
        B = T * N_
        if B % MB != 0:                                                  # the reference's reshape raises here (:329)
            raise ValueError(f"cannot reshape array of size {E * B} into shape ({E},{MB},{B // MB})")
        M = B // MB
        self._resync_optimizer()
        h_idx = [torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(E)]
        worker = _PermWorker(B, E, MB, [h.numpy() for h in h_idx])
        worker.start()
        # GAE with the values stored at rollout time, returns, advantage normalisation (recurrent_ppo.py:315-318)
        stats = torch.zeros(2, dtype=torch.float64, device=dev)
        adv = torch.empty(T, N_, device=dev)
        ret = torch.empty(T, N_, device=dev)
        ctx.gae(ro.rewards, ro.terminations, ro.truncations, ro.values.contiguous(), ro.next_values.contiguous(), cfg.gamma,
                cfg.gae_lambda, advantages=adv, returns=ret, stats=stats)
        # env-sharded data parallelism (rank r holds envs [r N, (r+1) N) of the global rollout; the sequences shard with no halo):
        # global advantage statistics, loss means over the global minibatch, gradients summed over the ranks before the clip
        dist.all_reduce_sum(stats)
        if cfg.advantage_norm:
            adv = ctx.adv_normalize(adv, stats, B * dist.world)
        hyper = self._hyper(cfg, M * dist.world, B * dist.world)
        hyper.advantage_norm = 0                                         # already normalised above
        old_logp, adv_f, ret_f = ro.log_probs.reshape(B).contiguous(), adv.view(B), ret.view(B)
        if self.continuous:
            A = ro.actions.shape[-1]
            act_bits = ro.actions.reshape(B, A).contiguous()
        else:
            act_bits = ro.actions.reshape(B).to(torch.int32).view(torch.float32)
            A = net.actor_out_layer.out_features
        losses = torch.zeros(E * MB, 4, device=dev)
        loss_ws = torch.empty(ctx.ppo_loss_workspace_bytes(M, max(A, 32)) // 4 + 64, device=dev)
        idx = torch.empty(E, B, dtype=torch.int32, device=dev)
        hx0 = ro.hx0.clone()
        for e in range(E):
            worker.wait(e)
            idx[e].copy_(h_idx[e], non_blocking=True)
            for k in range(MB):
                mb = idx[e][k * M:(k + 1) * M]
                mb64 = mb.to(torch.int64)
                a_mb = ctx.gather_rows(act_bits, mb)
                lp_mb, adv_mb, ret_mb = ctx.gather_rows(old_logp, mb), ctx.gather_rows(adv_f, mb), ctx.gather_rows(ret_f, mb)
                self.adam_step += 1
                hyper.step = self.adam_step
                self.G.zero_()
                # full-sequence forward with the current parameters, then the minibatch rows (recurrent_ppo.py:337-341)
                if self.continuous:
                    means, log_stds, values, _ = net.get_means_log_stds_values_and_hx(ro.obs, hx0, ro.prev_dones)
                    mean_mb = means.reshape(B, A).index_select(0, mb64).contiguous()
                    ls_mb = log_stds.reshape(B, A).index_select(0, mb64).contiguous()
                    val_mb = values.reshape(B).index_select(0, mb64).contiguous()
                    dmean, dls, dval = torch.empty_like(mean_mb), torch.empty_like(ls_mb), torch.empty_like(val_mb)
                    ctx.ppo_loss_gaussian(mean_mb.detach(), ls_mb.detach(), val_mb.detach(), a_mb, lp_mb, adv_mb, ret_mb, hyper,
                                          losses[e * MB + k], dmean, dls, dval, loss_ws, log_std_row_stride=A)
                    torch.autograd.backward([mean_mb, ls_mb, val_mb], [dmean, dls, dval])
                else:
                    logits, values, _ = net.get_logits_values_and_hx(ro.obs, hx0, ro.prev_dones)
                    logits_mb = logits.reshape(B, A).index_select(0, mb64).contiguous()
                    val_mb = values.reshape(B).index_select(0, mb64).contiguous()
                    dlogits, dval = torch.empty_like(logits_mb), torch.empty_like(val_mb)
                    ctx.ppo_loss_discrete(logits_mb.detach(), val_mb.detach(), a_mb.view(torch.int32), lp_mb, adv_mb, ret_mb, hyper,
                                          losses[e * MB + k], dlogits, dval, loss_ws)
                    torch.autograd.backward([logits_mb, val_mb], [dlogits, dval])
                if dist.enabled:
                    dist.all_reduce_sum(self.G)
                    dist.all_reduce_sum(losses[e * MB + k])
                ctx.clip_adam_step(self.P, self.G, self.M, self.V, hyper, self.adam_ws, self.grad_norm)
        worker.finish()
        self._publish_steps()
        self.last_losses = losses


def rnn_param_slices(desc: N.RnnDesc, lay: N.RnnLayout):
    """name (reference module naming, recurrent_ppo.py:101-125; RecurrentContinuousActorCriticNetwork's when desc.continuous)
    -> (offset, shape) in the flat buffers (dppo_rnn_layout)."""
    D, H, Hg, A = desc.obs_dim, desc.hidden, desc.gru_hidden, desc.act_dim
    actor = "actor_mean_head" if desc.continuous else "actor_head"
    s = {
        "base.0.weight": (lay.w1, (H, D)), "base.0.bias": (lay.b1, (H,)),
        "gru.weight_ih_l0": (lay.wih, (3 * Hg, H)), "gru.weight_hh_l0": (lay.whh, (3 * Hg, Hg)),
        "gru.bias_ih_l0": (lay.bih, (3 * Hg,)), "gru.bias_hh_l0": (lay.bhh, (3 * Hg,)),
        f"{actor}.0.weight": (lay.w3, (H, Hg)), f"{actor}.0.bias": (lay.b3, (H,)),
        f"{actor}.2.weight": (lay.wa, (A, H)), f"{actor}.2.bias": (lay.ba, (A,)),
        "critic_head.0.weight": (lay.w3 + H * Hg, (H, Hg)), "critic_head.0.bias": (lay.b3 + H, (H,)),
        "critic_head.2.weight": (lay.wc, (1, H)), "critic_head.2.bias": (lay.bc, (1,)),
    }
    if desc.continuous:
        s["actor_log_std"] = (lay.log_std, (1, A))
    return s


class FusedRecurrentEngine(_EngineBase):
    """learn() / forward of the default recurrent network on the libdppo kernels only (csrc/rnn.cu)."""

    fused = True

    def __init__(self, ctx, network, cfg, obs_dim, act_dim, device, dist: _Dist | None = None, continuous=False):
        self.ctx, self.cfg, self.device, self.continuous = ctx, cfg, device, continuous
        self.dist = dist if dist is not None else _Dist(None, False)
        self.network = network
        self.desc = N.RnnDesc(int(obs_dim), int(cfg.network_hidden_dim), int(cfg.gru_hidden_dim), int(act_dim), int(continuous))
        self.layout = N.rnn_layout(self.desc)
        self._adopt(network, rnn_param_slices(self.desc, self.layout), int(self.layout.total))
        # Gaussian policy: the actor_log_std [A] the sampling kernel reads (a view of the flat parameter buffer)
        self.log_std = self.P[self.layout.log_std:self.layout.log_std + int(act_dim)] if continuous else None
        self.last_losses = None
        self.draws = 0
        self.seed = self.dist.shared_seed(cfg.seed if cfg.seed is not None else (None if self.dist.enabled else int(np.random.randint(0, 2 ** 31 - 1))), device)
        self.env_offset = self.dist.rank * cfg.num_envs              # global id of this shard's first environment (sampling keys)
        self._ws = {}
        self._bufs = {}
        self._seen_keys = []
        self.use_graphs = True

    def _workspace(self, T, N_, M, training):
        key = (T, N_, M, bool(training))
        if key not in self._ws:
            self._ws[key] = torch.empty(self.ctx.rnn_workspace_bytes(self.desc, T, N_, M, training) // 4 + 64, device=self.device)
        return self._ws[key]

    def forward(self, obs, hx, prev_dones, heads=3):
        """(logits [T,N,A], values [T,N], hx [1,N,Hg]) of get_logits_values_and_hx / get_values (recurrent_ppo.py:127-149); with
        a Gaussian policy the first output holds the action means."""
        T, N_ = obs.shape[:2]
        dev, A, Hg = self.device, self.desc.act_dim, self.desc.gru_hidden
        logits = torch.empty(T, N_, A, device=dev) if heads & 1 else None
        values = torch.empty(T, N_, device=dev) if heads & 2 else None
        hx_out = torch.empty(1, N_, Hg, device=dev)
        pd = None if prev_dones is None else prev_dones.to(torch.uint8).contiguous()
        self.ctx.rnn_forward(self.desc, self.P, obs.contiguous(), pd, None if hx is None else hx.contiguous(), T, N_, heads,
                             logits, values, hx_out, self._workspace(T, N_, T * N_, False))
        return logits, values, hx_out

    def _buffers(self, T, N_, E, MB):
        key = (T, N_, E, MB)
        b = self._bufs.get(key)
        if b is None:
            dev, B = self.device, T * N_
            b = self._bufs[key] = dict(
                stats=torch.zeros(2, dtype=torch.float64, device=dev), adv=torch.empty(T, N_, device=dev), ret=torch.empty(T, N_, device=dev),
                losses=torch.zeros(E * MB, 4, device=dev), idx=[torch.empty(B, dtype=torch.int32, device=dev) for _ in range(2)],
                h_sets=[[torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(E)] for _ in range(2)], h_set=0, h_consumed=[None, None],
                old_logp=torch.empty(B, device=dev),
                actions=torch.empty(B, self.desc.act_dim, device=dev) if self.continuous else torch.empty(B, dtype=torch.int32, device=dev),
                pd=torch.empty(T, N_, dtype=torch.uint8, device=dev), hx0=torch.empty(N_, self.desc.gru_hidden, device=dev),
                values=torch.empty(T, N_, device=dev), next_values=torch.empty(T, N_, device=dev),
                consts=[torch.zeros(MB, 4, dtype=torch.float32, device=dev) for _ in range(2)],
                h_consts=[torch.zeros(MB, 4, dtype=torch.float32).pin_memory() for _ in range(2)],
                consts_copied=[torch.cuda.Event() for _ in range(2)], g_losses=[torch.zeros(MB, 4, device=dev) for _ in range(2)],
                graphs={})
        return b

    def learn(self, ro: RecurrentRollout):
        cfg, ctx, dev, dist = self.cfg, self.ctx, self.device, self.dist
        T, N_ = ro.T, ro.N
        E, MB = cfg.num_epochs, cfg.num_minibatches
        B = T * N_
        if B % MB != 0:                                                  # the reference's reshape raises here (:329)
            raise ValueError(f"cannot reshape array of size {E * B} into shape ({E},{MB},{B // MB})")
        M = B // MB
        self._resync_optimizer()
        b = self._buffers(T, N_, E, MB)
        b["h_set"] ^= 1
        h_idx = b["h_sets"][b["h_set"]]
        if b["h_consumed"][b["h_set"]] is not None:
            b["h_consumed"][b["h_set"]].synchronize()                    # the async copies out of this pinned set are done
        worker = _PermWorker(B, E, MB, [h.numpy() for h in h_idx])
        worker.start()
        # learn()-persistent copies in the kernels' dtypes (stable addresses: the optimiser steps are replayed as a CUDA graph)
        b["old_logp"].copy_(ro.log_probs.reshape(B)); b["actions"].copy_(ro.actions.reshape(b["actions"].shape))
        b["pd"].copy_(ro.prev_dones); b["hx0"].copy_(ro.hx0.reshape(N_, -1))
        b["values"].copy_(ro.values); b["next_values"].copy_(ro.next_values)
        # GAE with the values stored at rollout time + returns + advantage sums (recurrent_ppo.py:315-318); the normalisation
        # itself is applied while the head kernel gathers the advantages
        stats, adv, ret = b["stats"], b["adv"], b["ret"]
        stats.zero_()
        ctx.gae(ro.rewards, ro.terminations, ro.truncations, b["values"], b["next_values"], cfg.gamma, cfg.gae_lambda, advantages=adv,
                returns=ret, stats=stats)
        # Env-sharded data parallelism: rank r holds envs [r N, (r+1) N) of the global rollout.  The GRU sequences shard by
        # environment with no halo, so forward / BPTT scans stay rank-local; what is global: the advantage statistics, the loss
        # means (global minibatch = the ranks' local minibatches side by side, rank-local permutations) and the gradient, summed
        # over the ranks with NCCL before the global-norm clip (recurrent_ppo.py:362).
        dist.all_reduce_sum(stats)
        hyper = self._hyper(cfg, M * dist.world, B * dist.world)
        if not dist.enabled:
            hyper.grad_sumsq = self.grad_sumsq.data_ptr()            # gradient assembly leaves the norm partials for the Adam kernel
        losses = b["losses"]
        ws = self._workspace(T, N_, M, True)

        def step(idx_k, losses_k):
            ctx.rnn_grad_minibatch(self.desc, self.P, self.G, ro.obs, b["pd"], b["hx0"], T, N_, b["actions"], b["old_logp"], adv.view(B),
                                   ret.view(B), stats, idx_k, M, hyper, losses_k, ws)
            if dist.enabled:
                dist.all_reduce_sum(self.G)
                dist.all_reduce_sum(losses_k)
            ctx.clip_adam_step(self.P, self.G, self.M, self.V, hyper, self.adam_ws, self.grad_norm)

        # From the second learn() on the same rollout buffers the MB optimiser steps of an epoch (15 launches each) are replayed as
        # one CUDA graph; the minibatch indices and Adam's two step-dependent constants are device-resident (like the MLP engine).
        key = (ro.obs.data_ptr(), ro.rewards.data_ptr(), T, N_, E, MB, cfg.ppo_clip, cfg.value_loss_weight, cfg.entropy_beta,
               cfg.grad_norm_clip, cfg.adam_eps, bool(cfg.advantage_norm))
        use_graph = self.use_graphs and key in self._seen_keys and not dist.enabled     # (NCCL calls are not captured)
        if key not in self._seen_keys:
            self._seen_keys = (self._seen_keys + [key])[-4:]
        gs = None
        if use_graph:
            gs = b["graphs"].get(key)
            if gs is None:
                if len(b["graphs"]) >= 4:
                    b["graphs"].pop(next(iter(b["graphs"])))
                gs = b["graphs"][key] = []
                cap = torch.cuda.Stream()
                cap.wait_stream(torch.cuda.current_stream())
                for p in range(2):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=cap):
                        for k in range(MB):
                            hyper.step = 1
                            hyper.step_consts = b["consts"][p][k].data_ptr()
                            step(b["idx"][p][k * M:(k + 1) * M], b["g_losses"][p][k])
                    gs.append(g)
                hyper.step_consts = None
                torch.cuda.current_stream().wait_stream(cap)
        b1, b2 = hyper.beta1, hyper.beta2
        for e in range(E):
            p = e & 1
            worker.wait(e)
            b["idx"][p].copy_(h_idx[e], non_blocking=True)               # stream-ordered after the steps that last read idx[p]
            b["h_consumed"][b["h_set"]] = torch.cuda.Event()
            b["h_consumed"][b["h_set"]].record()
            if gs is not None:
                b["consts_copied"][p].synchronize()
                hc = b["h_consts"][p].numpy()
                for k in range(MB):
                    st = self.adam_step + k + 1                          # torch/optim/adam.py:531-547, python-float bias corrections
                    hc[k, 0] = np.float32(np.sqrt(1.0 - b2 ** st))
                    hc[k, 1] = np.float32(-(hyper.lr / (1.0 - b1 ** st)))
                b["consts"][p].copy_(b["h_consts"][p], non_blocking=True)
                b["consts_copied"][p].record()
                gs[p].replay()
                losses[e * MB:(e + 1) * MB].copy_(b["g_losses"][p])
                self.adam_step += MB
                continue
            for k in range(MB):
                self.adam_step += 1
                hyper.step = self.adam_step
                step(b["idx"][p][k * M:(k + 1) * M], losses[e * MB + k])
        worker.finish()
        self._publish_steps()
        self.last_losses = losses


class RecurrentPPO(PolicyEvaluation):
    """Recurrent (GRU) discrete-action PPO (reference: diamond/recurrent_ppo.py:164-394)."""
    _continuous = False
    _recurrent = True
    _default_network: Any = RecurrentActorCriticNetwork

    def __init__(self, env_fn: Callable[[], Any], cfg: RecurrentPPOConfig = RecurrentPPOConfig(),
                 network_cls: Any = RecurrentActorCriticNetwork, *, process_group=None, dp: bool = False) -> None:
        """process_group / dp (additive): env-sharded data parallelism, one process per GPU -- this rank simulates and learns from
        cfg.num_envs of the world_size * cfg.num_envs environments (rank-local minibatch permutations, NCCL gradient sum)."""
        self.device = _require_cuda()
        self.ctx = N.get_context(self.device.index)
        if cfg.seed is not None:
            np.random.seed(cfg.seed)                                    # recurrent_ppo.py:173-175
            torch.manual_seed(cfg.seed)
        self._dist = _Dist(process_group, dp, "local", "nccl", "numpy")
        self._env_fn = env_fn                                            # evaluate() builds new environments from it
        if getattr(env_fn, "vectorized", False):
            self.envs = env_fn(cfg.num_envs)
            if self._dist.enabled and getattr(self.envs, "device_resident", False) and self.envs.desc.env_offset == 0:
                self.envs.desc.env_offset = self._dist.rank * cfg.num_envs      # distinct reset / dynamics draws per shard
        else:
            self.envs = gym.vector.SyncVectorEnv([env_fn for _ in range(cfg.num_envs)], copy=True, autoreset_mode="Disabled")
        obs_space, act_space = self.envs.single_observation_space, self.envs.single_action_space
        self.network = network_cls(obs_space, act_space, cfg=cfg).to(self.device)
        # touches nn.Linear only (:152-161); no 0.01-gain output layer for the Gaussian policy (continuous_ppo.py:114-121)
        network_parameter_init_(self.network, gain=sqrt(2.0), small_actor_out=not self._continuous)
        if self._dist.enabled:                                           # replicas start from rank 0's parameters
            for p in self.network.parameters():
                self._dist.dist.broadcast(p.data, src=0, group=self._dist.group)
        self.obs_dim = int(np.prod(obs_space.shape))
        self.act_dim = int(np.prod(act_space.shape)) if self._continuous else int(act_space.n)
        if type(self.network) is self._default_network:                  # default network: libdppo kernels end to end
            self.engine = FusedRecurrentEngine(self.ctx, self.network, cfg, self.obs_dim, self.act_dim, self.device, self._dist,
                                               self._continuous)
        else:                                                            # custom network_cls: the module runs under autograd
            self.engine = RecurrentEngine(self.ctx, self.network, cfg, self.device, self._dist, self._continuous)
        self.optimizer = torch.optim.Adam(self.network.parameters(), lr=cfg.lr, eps=cfg.adam_eps)
        self.engine.bind_optimizer(self.optimizer)
        self.lr_scheduler = torch.optim.lr_scheduler.LinearLR(
            self.optimizer, start_factor=1.0, end_factor=0.05 if cfg.decay_lr else 1.0,
            total_iters=cfg.total_steps // (cfg.num_envs * cfg.rollout_steps))
        self.logger = Logger()
        self.timer = Timer()
        self.checkpointer = Checkpointer(folder="models", run_name="default")
        self.ticker = Ticker(cfg.total_steps, cfg.num_envs, cfg.rollout_steps, verbose=cfg.verbose)
        self.cfg = cfg
        self._device_ro, self._epstats = None, None

    # device-side episode statistics (shared with the MLP agents)
    _device_episode_stats = _PPOBase._device_episode_stats
    _flush_episode_stats = _PPOBase._flush_episode_stats

    # ---- rollout (recurrent_ppo.py:205-263) ----------------------------------------------------------
    def rollout(self) -> RecurrentRollout:
        cfg, dev = self.cfg, self.device
        T, N_ = cfg.rollout_steps, cfg.num_envs
        if getattr(self.envs, "device_resident", False) and getattr(self.engine, "fused", False):
            return self._rollout_device()
        cont = self._continuous
        ro = RecurrentRollout(T, N_, self.obs_dim, cfg.gru_hidden_dim, dev, self.act_dim if cont else None)
        observations, hx, prev_dones = self.current_observations, self.current_hx, self.prev_dones
        ro.hx0.copy_(hx)
        for t in range(T):
            obs_t = torch.as_tensor(np.asarray(observations, dtype=np.float32)[None, ...], device=dev)
            pd_t = torch.as_tensor(np.asarray(prev_dones)[None, ...], dtype=torch.bool, device=dev)
            log_std = None
            if getattr(self.engine, "fused", False):
                logits, values, new_hx = self.engine.forward(obs_t, hx, pd_t)
                log_std = self.engine.log_std
            elif cont:
                with torch.inference_mode():
                    logits, ls, values, new_hx = self.network.get_means_log_stds_values_and_hx(obs_t, hx, pd_t)
                    ls = ls.reshape(N_, -1)
                    log_std = ls[0].contiguous() if bool((ls == ls[:1]).all()) else ls   # shared [A] vector, else per row
            else:
                with torch.inference_mode():
                    logits, values, new_hx = self.network.get_logits_values_and_hx(obs_t, hx, pd_t)
            if cont and log_std.dim() == 1:
                # JointNormal(mean, exp(log_std)).sample() + log_prob on the device (counter-based generator, dppo_sample_gaussian)
                actions = torch.empty(N_, self.act_dim, device=dev)
                self.ctx.sample_gaussian(logits.reshape(N_, -1).contiguous(), log_std, self.engine.seed, self.engine.draws,
                                         self.engine.env_offset, actions, ro.log_probs[t])
            elif cont:                                                   # state-dependent std of a custom network
                dist_t = torch.distributions.Normal(logits.reshape(N_, -1), log_std.exp())
                actions = dist_t.sample()
                ro.log_probs[t].copy_(dist_t.log_prob(actions).sum(-1))
            else:
                # Categorical(logits).sample() + log_prob on the device (counter-based generator, dppo_sample_categorical)
                actions = torch.empty(N_, dtype=torch.int64, device=dev)
                self.ctx.sample_categorical(logits.squeeze(0).contiguous(), self.engine.seed, self.engine.draws, self.engine.env_offset, actions, ro.log_probs[t])
            self.engine.draws += 1
            next_observations, rewards, terminations, truncations, infos = self.envs.step(actions.cpu().numpy())
            tick_rewards = infos.get("raw_rewards", rewards) if isinstance(infos, dict) else rewards   # raw, if the env normalises
            final_t = torch.as_tensor(np.asarray(next_observations, dtype=np.float32)[None, ...], device=dev)
            if getattr(self.engine, "fused", False):
                _, next_values, _ = self.engine.forward(final_t, new_hx, None, heads=2)
            else:
                with torch.inference_mode():
                    next_values = self.network.get_values(final_t, new_hx, None)  # V(final obs | h_{t+1}), no reset (:226-232)
            ro.obs[t].copy_(obs_t.squeeze(0)); ro.actions[t].copy_(actions)
            ro.rewards[t].copy_(torch.as_tensor(np.asarray(rewards, dtype=np.float32), device=dev))
            ro.terminations[t].copy_(torch.as_tensor(np.asarray(terminations, dtype=np.float32), device=dev))
            ro.truncations[t].copy_(torch.as_tensor(np.asarray(truncations, dtype=np.float32), device=dev))
            ro.prev_dones[t].copy_(pd_t.squeeze(0)); ro.values[t].copy_(values.squeeze(0)); ro.next_values[t].copy_(next_values.squeeze(0))
            dones = np.logical_or(terminations, truncations)
            if np.any(dones):
                observations, infos = self.envs.reset(options={"reset_mask": dones})
            else:
                observations = next_observations
            hx = new_hx
            prev_dones = dones
            if self.ticker is not None:
                self.ticker.tick(tick_rewards, dones)
        ro.filled = T
        self.current_observations, self.current_hx, self.prev_dones = observations, hx, prev_dones
        return ro

    def _rollout_device(self) -> RecurrentRollout:
        """Device-resident environments (diamond.envs.DeviceVectorEnv): the whole rollout loop of recurrent_ppo.py:214-263 stays on
        the GPU -- GRU step, sampling kernel, environment kernel (which writes row t of the rollout tensors and resets finished
        environments), V(final observation | h_{t+1}) -- with no PCIe crossing and no host synchronisation; the rollout tensors are
        persistent, so learn() replays its optimiser steps as CUDA graphs.  Episode statistics: dppo_episode_stats, read lazily."""
        cfg, dev, envs, eng, ctx = self.cfg, self.device, self.envs, self.engine, self.ctx
        T, N_ = cfg.rollout_steps, cfg.num_envs
        A, Hg = eng.desc.act_dim, eng.desc.gru_hidden
        ro = self._device_ro
        cont = self._continuous
        if ro is None:
            ro = self._device_ro = RecurrentRollout(T, N_, self.obs_dim, cfg.gru_hidden_dim, dev, A if cont else None)
            ro.next_obs = torch.empty(T, N_, self.obs_dim, device=dev)
            # rewards are normalised: the raw ones feed the Ticker
            ro.raw_rewards = torch.empty(T, N_, device=dev) if getattr(envs, "normalize_reward", False) else None
            ro.pd_u8 = torch.zeros(N_, dtype=torch.uint8, device=dev)
            ro.actions_dev = torch.empty(N_, A, device=dev) if cont else torch.empty(N_, dtype=torch.int64, device=dev)
            ro.pd_f32, ro.pd_bool = torch.empty(N_, device=dev), torch.zeros(N_, dtype=torch.bool, device=dev)
            ro.logits, ro.val1, ro.nv1 = torch.empty(N_, A, device=dev), torch.empty(N_, device=dev), torch.empty(N_, device=dev)
            ro.hx_buf = [torch.zeros(N_, Hg, device=dev) for _ in range(3)]      # [0], [1]: ping-pong state; [2]: discarded output
            ro.ws1 = eng._workspace(1, N_, N_, False)
            self._ro_graph, self._ro_seen = None, 0
        if not torch.is_tensor(self.prev_dones):
            ro.pd_u8.copy_(torch.as_tensor(np.asarray(self.prev_dones, dtype=np.uint8)))
        if self.current_hx.data_ptr() != ro.hx_buf[0].data_ptr():
            ro.hx_buf[0].copy_(self.current_hx.reshape(N_, Hg))
        ro.hx0.copy_(ro.hx_buf[0].reshape(ro.hx0.shape))

        def steps(counter_of):
            for t in range(T):
                hx, new_hx = ro.hx_buf[t & 1], ro.hx_buf[(t + 1) & 1]
                ro.prev_dones[t].copy_(ro.pd_u8)
                ctx.rnn_forward(eng.desc, eng.P, envs.cur_obs, ro.pd_u8, hx, 1, N_, 3, ro.logits, ro.val1, new_hx, ro.ws1)
                if cont:                                                 # ro.logits holds the action means
                    ctx.sample_gaussian(ro.logits, eng.log_std, eng.seed, counter_of(t), eng.env_offset, ro.actions_dev, ro.log_probs[t])
                else:
                    ctx.sample_categorical(ro.logits, eng.seed, counter_of(t), eng.env_offset, ro.actions_dev, ro.log_probs[t])
                ro.actions[t].copy_(ro.actions_dev)
                ro.values[t].copy_(ro.val1)
                # environment kernel: writes obs[t] (the observation acted on), next_obs[t] (true final observation), rewards, masks;
                # finished environments are reset in the same kernel
                ctx.env_step(envs.desc, envs._st, ro.actions_dev, t, True, ro.obs, ro.next_obs, None, ro.rewards, ro.terminations,
                             ro.truncations, raw_rewards=ro.raw_rewards)
                # V(final observation | h_{t+1}): one more GRU step from the post-step state, no reset (recurrent_ppo.py:226-232)
                ctx.rnn_forward(eng.desc, eng.P, ro.next_obs[t], None, new_hx, 1, N_, 2, None, ro.nv1, ro.hx_buf[2], ro.ws1)
                ro.next_values[t].copy_(ro.nv1)
                torch.add(ro.terminations[t], ro.truncations[t], out=ro.pd_f32)
                torch.gt(ro.pd_f32, 0, out=ro.pd_bool)
                ro.pd_u8.copy_(ro.pd_bool)                               # dones of step t = prev_dones of step t + 1 (:259-261)
            if T & 1:                                                    # the state always ends in hx_buf[0]
                ro.hx_buf[0].copy_(ro.hx_buf[1])

        # From the third rollout the T x 14 launches are replayed as ONE CUDA graph; the sampling draw counters baked into it are
        # relative to a device-resident base (dppo_set_draw_counter_base), so every replay draws fresh numbers.
        if self._ro_graph is not None:
            self._ro_graph["base"].fill_(eng.draws)
            self._ro_graph["graph"].replay()
        elif eng.use_graphs and self._ro_seen >= 2:
            base = torch.zeros(1, dtype=torch.int64, device=dev)
            graph = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            ctx.set_draw_counter_base(base)
            try:
                with torch.cuda.graph(graph):
                    steps(lambda t: t)
            finally:
                ctx.set_draw_counter_base(None)
            self._ro_graph = dict(graph=graph, base=base)
            base.fill_(eng.draws)
            graph.replay()
        else:
            self._ro_seen += 1
            steps(lambda t: eng.draws + t)
        eng.draws += T
        ro.filled = T
        if self.ticker is not None:
            self._device_episode_stats(ro)
        self.current_observations, self.current_hx, self.prev_dones = envs.cur_obs, ro.hx_buf[0].reshape(1, N_, Hg), ro.pd_u8
        return ro

    # ---- evaluation (diamond/evaluation.py) --------------------------------------------------------------------------------
    def predict(self, observations, hx=None, dones=None, deterministic: bool = True):
        """One step of the current policy: observations [n, obs_dim], hidden state hx [1, n, Hg] (None: zeros) and dones [n] (None:
        no resets; True zeroes the hidden state of that environment before the step, as prev_dones in a rollout).  Returns
        (actions, new_hx): NumPy arrays for host observations, device tensors for device tensors.  deterministic=True: the first
        argmax of the logits or the Gaussian means (not clipped); False: a draw of the evaluation generator, which leaves the
        training sampling counter and the numpy / torch streams alone.  The default network runs dppo_rnn_forward and the greedy /
        sampling kernels; a custom network_cls its get_logits_values_and_hx / get_means_log_stds_values_and_hx under inference_mode."""
        dev, Hg = self.device, self.cfg.gru_hidden_dim
        obs = as_device_obs(observations, self.obs_dim, dev)
        n = obs.shape[0]
        h = torch.zeros(1, n, Hg, device=dev) if hx is None else as_device_obs(hx, Hg, dev).reshape(1, n, Hg)
        pd = None if dones is None else torch.as_tensor(np.asarray(dones) if not torch.is_tensor(dones) else dones).to(dev, torch.bool).reshape(1, n)
        eng, log_std = self.engine, None
        if getattr(eng, "fused", False):
            head, _, new_hx = eng.forward(obs.reshape(1, n, -1), h, pd, heads=1)
            log_std = eng.log_std
        else:
            with torch.inference_mode():
                if self._continuous:
                    head, log_stds, _, new_hx = self.network.get_means_log_stds_values_and_hx(obs.reshape(1, n, -1), h, pd)
                    log_std = shared_log_std(log_stds.reshape(n, -1))
                else:
                    head, _, new_hx = self.network.get_logits_values_and_hx(obs.reshape(1, n, -1), h, pd)
        head = head.reshape(n, -1).contiguous()
        key, counter = self._eval_draw() if not deterministic else (0, 0)
        actions = select_actions(self.ctx, head, log_std, deterministic, key, counter, greedy_kernel=getattr(eng, "fused", False))
        new_hx = new_hx.reshape(1, n, Hg).clone()
        if torch.is_tensor(observations):
            return actions, new_hx
        return actions.cpu().numpy(), new_hx.cpu().numpy()

    # ---- GAE (recurrent_ppo.py:265-299) ----------------------------------------------------------------
    def calculate_advantage(self, rewards, terminations, truncations, values, next_values) -> torch.Tensor:
        args = [torch.as_tensor(x).to(self.device, torch.float32).contiguous() for x in
                (rewards, terminations, truncations, values, next_values)]
        return self.ctx.gae(*args, self.cfg.gamma, self.cfg.gae_lambda)

    # ---- learn (recurrent_ppo.py:301-367) ---------------------------------------------------------------
    def learn(self, experience) -> None:
        ro = experience if isinstance(experience, RecurrentRollout) else RecurrentRollout.from_lists(experience, self.device, self._continuous)
        self.engine.learn(ro)
        self.optimizer._opt_called = True
        self.lr_scheduler.step()

    @property
    def last_losses(self):
        return self.engine.last_losses

    # ---- train (recurrent_ppo.py:369-394) ---------------------------------------------------------------
    def train(self) -> None:
        cfg = self.cfg
        seed = cfg.seed                                                # shards are different environments of one global run
        if seed is not None and self._dist.enabled and not getattr(self.envs, "device_resident", False):
            seed = cfg.seed + self._dist.rank * cfg.num_envs
        self.current_observations, _ = self.envs.reset(seed=seed)
        self.prev_dones = np.zeros(cfg.num_envs, dtype=bool)
        self.current_hx = torch.zeros(1, cfg.num_envs, cfg.gru_hidden_dim, device=self.device)
        if self._epstats is not None:                                  # fresh environments: running returns / lengths restart
            self._flush_episode_stats()
            self._epstats["ep_return"].zero_()
            self._epstats["ep_len"].zero_()
        last_checkpoint_time = time.time()
        total_rollouts = cfg.total_steps // (cfg.rollout_steps * cfg.num_envs)
        env_steps = 0
        for rollout_idx in range(total_rollouts):
            experience = self.rollout()
            self.learn(experience)
            env_steps = (rollout_idx + 1) * cfg.rollout_steps * cfg.num_envs
            if cfg.checkpoint and self._dist.rank == 0 and time.time() - last_checkpoint_time >= cfg.save_interval:
                self.checkpointer.save(env_steps, self.network, self.optimizer)      # replicas are identical: rank 0 writes
                last_checkpoint_time = time.time()
        if cfg.checkpoint and total_rollouts > 0 and self._dist.rank == 0:
            self.checkpointer.save(env_steps, self.network, self.optimizer)
        self._flush_episode_stats()
        self.envs.close()


class RecurrentContinuousPPO(RecurrentPPO):
    """Recurrent (GRU) Gaussian-policy PPO for Box action spaces: RecurrentPPO with the actor of ContinuousPPO
    (continuous_ppo.py:50-121: mean head, state-independent log-std, actions neither squashed nor clipped)."""
    _continuous = True
    _default_network = RecurrentContinuousActorCriticNetwork

    def __init__(self, env_fn: Callable[[], Any], cfg: RecurrentContinuousPPOConfig = RecurrentContinuousPPOConfig(),
                 network_cls: Any = RecurrentContinuousActorCriticNetwork, *, process_group=None, dp: bool = False) -> None:
        super().__init__(env_fn, cfg, network_cls, process_group=process_group, dp=dp)
