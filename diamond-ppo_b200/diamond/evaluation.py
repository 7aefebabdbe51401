"""Policy evaluation for the four agents: `predict()` helpers and `evaluate()`.

`evaluate(num_episodes)` plays the policy (greedy by default) on NEW environment instances and returns the return and length of
every finished episode.  Episodes are split over the environments as Stable-Baselines3's `evaluate_policy` splits them: environment
i runs its first (num_episodes + i) // num_envs episodes, so short episodes are not favoured the way "the first K episodes to
finish" would favour them.  Results are ordered by (environment, episode).

Arithmetic (the same in both loops below, and in dppo_eval_episodes): per environment the running return is the sum, in float64,
of the raw rewards the environment hands out (a normalising device environment's raw-reward row, float32 widened to float64), the
length counts steps, and an episode ends on termination | truncation.

Two loops run it:
  * device environments with a default network: chunks of EVAL_CHUNK steps, each step fused forward -> greedy kernel (or the
    means, or a sampling kernel) -> environment kernel with in-kernel resets, then one dppo_eval_episodes launch per chunk.  The
    one host synchronisation per chunk is the copy of the number of environments still short of their quota.  From the second
    chunk on, a chunk is replayed as a CUDA graph.
  * host environments, and custom networks on any environment: a host loop over `predict` with masked resets.

Under data parallelism evaluation is rank-local: each rank evaluates on its own new environments; nothing is exchanged.
"""
from __future__ import annotations

import numpy as np
import torch

EVAL_CHUNK = 64           # steps per device chunk (even: the recurrent hidden state ping-pongs between two buffers)
DEFAULT_MAX_STEPS = 100_000


def episode_quotas(num_episodes: int, num_envs: int) -> np.ndarray:
    """Episodes environment i must record: (num_episodes + i) // num_envs (Stable-Baselines3's evaluate_policy split)."""
    return np.array([(num_episodes + i) // num_envs for i in range(num_envs)], dtype=np.int32)


def eval_key(seed: int) -> int:
    """Key of the evaluation generator (dppo_sample_* with draw counters that belong to evaluation): a function of the evaluation
    seed only, distinct from the key the training rollouts sample with."""
    return (int(seed) * 0x9E3779B97F4A7C15 + 0xD1B54A32D192ED03) % (1 << 64)


def select_actions(ctx, head, log_std, deterministic, key, counter, out=None, greedy_kernel=True):
    """Actions from the policy head [n, A].  log_std None: categorical logits; else Gaussian means with a shared log-std [A] or
    per-row log-stds [n, A].  Deterministic: the first argmax (greedy kernel, or torch.argmax for a custom module) or the means;
    else a draw of the evaluation generator (key, counter)."""
    if log_std is None:
        if deterministic:
            return ctx.select_greedy_categorical(head, out) if greedy_kernel else torch.argmax(head, -1)
        return ctx.sample_categorical(head, key, counter, 0, out)
    if deterministic:
        return head
    if log_std.dim() == 1:
        return ctx.sample_gaussian(head, log_std, key, counter, 0, out)
    g = torch.Generator(device=head.device)                         # state-dependent std of a custom module
    g.manual_seed((key ^ (counter * 0x9E3779B97F4A7C15)) % (1 << 63))
    return torch.normal(head, log_std.exp(), generator=g)


def shared_log_std(log_stds: torch.Tensor) -> torch.Tensor:
    """[n, A] log-stds of a custom Gaussian module -> the shared [A] vector when every row holds the same values, else [n, A]."""
    ls = log_stds.reshape(log_stds.shape[0], -1)
    return ls[0].contiguous() if bool((ls == ls[:1]).all()) else ls.contiguous()


def as_device_obs(observations, obs_dim: int, device) -> torch.Tensor:
    obs = observations if torch.is_tensor(observations) else torch.as_tensor(np.asarray(observations, dtype=np.float32))
    return obs.to(device, torch.float32).reshape(-1, obs_dim).contiguous()


class _MlpDevicePolicy:
    """One step of the default MLP on the device environments' current observations."""

    def __init__(self, agent, n):
        eng = agent.engine
        self.ctx, self.eng, self.n = agent.ctx, eng, n
        self.head = torch.empty(n, eng.A, dtype=torch.float32, device=agent.device)
        self.log_std = eng.P[eng.fm.layout.log_std:eng.fm.layout.log_std + eng.A] if eng.continuous else None
        self.out = (torch.empty(n, eng.A, dtype=torch.float32, device=agent.device) if eng.continuous
                    else torch.empty(n, dtype=torch.int64, device=agent.device))

    def act(self, obs, t, deterministic, key, counter):
        self.ctx.mlp_forward(self.eng.fm.desc, self.eng.P, obs, self.n, 1, self.head, None, self.eng.fwd_ws)
        return select_actions(self.ctx, self.head, self.log_std, deterministic, key, counter, self.out)

    def observe(self, term_t, trunc_t):
        pass


class _RnnDevicePolicy:
    """One step of the default GRU network, carrying the hidden state and the prev_dones resets as RecurrentPPO's device rollout."""

    def __init__(self, agent, n):
        eng, dev = agent.engine, agent.device
        self.ctx, self.eng, self.n = agent.ctx, eng, n
        A, Hg = eng.desc.act_dim, eng.desc.gru_hidden
        self.head = torch.empty(n, A, dtype=torch.float32, device=dev)
        self.log_std = eng.log_std
        self.out = torch.empty(n, A, dtype=torch.float32, device=dev) if eng.continuous else torch.empty(n, dtype=torch.int64, device=dev)
        self.hx = [torch.zeros(n, Hg, dtype=torch.float32, device=dev) for _ in range(2)]
        self.pd_u8 = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.pd_f32, self.pd_bool = torch.empty(n, device=dev), torch.zeros(n, dtype=torch.bool, device=dev)
        self.ws = eng._workspace(1, n, n, False)

    def act(self, obs, t, deterministic, key, counter):
        self.ctx.rnn_forward(self.eng.desc, self.eng.P, obs, self.pd_u8, self.hx[t & 1], 1, self.n, 1, self.head, None,
                             self.hx[(t + 1) & 1], self.ws)
        return select_actions(self.ctx, self.head, self.log_std, deterministic, key, counter, self.out)

    def observe(self, term_t, trunc_t):
        torch.add(term_t, trunc_t, out=self.pd_f32)                  # dones of step t = prev_dones of step t + 1
        torch.gt(self.pd_f32, 0, out=self.pd_bool)
        self.pd_u8.copy_(self.pd_bool)


def _unfinished(rec, quotas) -> list:
    return [int(e) for e in np.flatnonzero(np.asarray(rec) < quotas)]


class PolicyEvaluation:
    """evaluate() of the four agents.  The agent provides `predict`, `_env_fn`, `envs`, `engine`, `ctx`, `device`, `cfg` and the
    class attribute `_recurrent`."""

    _recurrent = False

    def _eval_generator(self) -> dict:
        g = getattr(self, "_eval_gen", None)
        if g is None:
            g = self._eval_gen = dict(key=eval_key(self.cfg.seed or 0), draws=0)
        return g

    def _eval_draw(self) -> tuple[int, int]:
        g = self._eval_generator()
        key, counter = g["key"], g["draws"]
        g["draws"] += 1
        return key, counter

    def _default_eval_seed(self) -> int:
        """Differs from the training environments' seed, so evaluation does not replay the training resets."""
        base = int(self.envs.desc.seed) if getattr(self.envs, "device_resident", False) else int(self.cfg.seed or 0)
        return (base + 0x9E3779B9) % (1 << 32)

    def evaluate(self, num_episodes: int = 10, *, num_envs: int | None = None, env_fn=None, seed: int | None = None,
                 deterministic: bool = True, max_steps: int = DEFAULT_MAX_STEPS) -> dict:
        """Plays the policy on new environments and returns {"returns": float64 [num_episodes], "lengths": int64 [num_episodes],
        "mean_return", "mean_length"}, ordered by (environment, episode).

        num_envs (default cfg.num_envs) environments from env_fn (default: the agent's own factory) are created and reset with
        `seed` (default: a value derived from, and different from, the training environments' seed); environment i records its
        first (num_episodes + i) // num_envs episodes.  deterministic=True plays the greedy policy (argmax / Gaussian means);
        False samples from a generator of evaluation's own, keyed by the seed.  Neither the training environments, their
        normalisation statistics, the training sampling counter nor the numpy / torch random streams are touched.  Normalising
        device environments evaluate with frozen copies of the training statistics (DeviceVectorEnv.load_frozen_statistics).
        max_steps bounds the steps per environment: an environment still short of its quota then raises a RuntimeError."""
        if num_episodes < 1:
            raise ValueError(f"num_episodes must be >= 1 (got {num_episodes})")
        num_envs = int(self.cfg.num_envs if num_envs is None else num_envs)
        if num_envs < 1:
            raise ValueError(f"num_envs must be >= 1 (got {num_envs})")
        env_fn = self._env_fn if env_fn is None else env_fn
        seed = self._default_eval_seed() if seed is None else int(seed)
        quotas = episode_quotas(int(num_episodes), num_envs)
        self._eval_gen = dict(key=eval_key(seed), draws=0)
        if getattr(env_fn, "vectorized", False):
            envs = env_fn(num_envs)
        else:
            from .agents import gym
            envs = gym.vector.SyncVectorEnv([env_fn for _ in range(num_envs)], copy=True, autoreset_mode="Disabled")
        try:
            device_env = getattr(envs, "device_resident", False)
            if device_env and envs.desc.normalize:
                envs.load_frozen_statistics(self.envs)
            if device_env and getattr(self.engine, "fused", False):
                returns, lengths = self._evaluate_device(envs, quotas, seed, deterministic, int(max_steps))
            else:
                returns, lengths = self._evaluate_host(envs, quotas, seed, deterministic, int(max_steps))
        finally:
            envs.close()
        return dict(returns=returns, lengths=lengths, mean_return=float(returns.mean()), mean_length=float(lengths.mean()))

    # ---- host loop over predict() ------------------------------------------------------------------------------------------
    def _evaluate_host(self, envs, quotas, seed, deterministic, max_steps):
        n = len(quotas)
        slots = np.concatenate([[0], np.cumsum(quotas)[:-1]]).astype(np.int64)
        out_ret, out_len = np.zeros(int(quotas.sum())), np.zeros(int(quotas.sum()), dtype=np.int64)
        ret, length, rec = np.zeros(n), np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
        remaining = int((quotas > 0).sum())
        obs, _ = envs.reset(seed=seed)
        hx, prev = None, np.zeros(n, dtype=bool)
        steps = 0
        while remaining > 0:
            if steps >= max_steps:
                raise RuntimeError(f"evaluate(): environments {_unfinished(rec, quotas)} did not finish their episodes within "
                                   f"max_steps={max_steps} steps")
            if self._recurrent:
                actions, hx = self.predict(obs, hx, prev, deterministic=deterministic)
            else:
                actions = self.predict(obs, deterministic=deterministic)
            next_obs, rewards, terms, truncs, infos = envs.step(actions)
            raw = infos.get("raw_rewards", rewards) if isinstance(infos, dict) else rewards
            ret += np.asarray(raw, dtype=np.float64)
            length += 1
            dones = np.logical_or(terms, truncs)
            for e in np.flatnonzero(dones):
                if rec[e] < quotas[e]:
                    out_ret[slots[e] + rec[e]], out_len[slots[e] + rec[e]] = ret[e], length[e]
                    rec[e] += 1
                    remaining -= int(rec[e] == quotas[e])
                ret[e], length[e] = 0.0, 0
            obs = envs.reset(options={"reset_mask": dones})[0] if np.any(dones) else next_obs
            prev = dones
            steps += 1
        return out_ret, out_len

    # ---- device loop: default networks on device environments ----------------------------------------------------------------
    def _evaluate_device(self, envs, quotas, seed, deterministic, max_steps):
        ctx, dev = self.ctx, self.device
        n, S, E = envs.num_envs, EVAL_CHUNK, int(quotas.sum())
        f = dict(dtype=torch.float32, device=dev)
        next_obs = torch.empty(S, n, envs.obs_dim, **f)
        rewards, terms, truncs = (torch.empty(S, n, **f) for _ in range(3))
        raw = torch.empty(S, n, **f) if envs.normalize_reward else None
        score = rewards if raw is None else raw
        slots = np.concatenate([[0], np.cumsum(quotas)[:-1]]).astype(np.int64)
        quota_d, slot_d = torch.as_tensor(quotas).to(dev), torch.as_tensor(slots).to(dev)
        ep_return = torch.zeros(n, dtype=torch.float64, device=dev)
        ep_len, recorded = torch.zeros(n, dtype=torch.int32, device=dev), torch.zeros(n, dtype=torch.int32, device=dev)
        out_ret, out_len = torch.zeros(E, dtype=torch.float64, device=dev), torch.zeros(E, dtype=torch.int32, device=dev)
        remaining = torch.tensor([int((quotas > 0).sum())], dtype=torch.int32, device=dev)
        h_rem = torch.zeros(1, dtype=torch.int32).pin_memory()
        policy = (_RnnDevicePolicy if self._recurrent else _MlpDevicePolicy)(self, n)
        gen = self._eval_generator()
        envs.reset(seed=seed)

        def chunk(T, counter_of):
            for t in range(T):
                a = policy.act(envs.cur_obs, t, deterministic, gen["key"], counter_of(t))
                ctx.env_step(envs.desc, envs._st, a, t, True, None, next_obs, None, rewards, terms, truncs, raw_rewards=raw)
                policy.observe(terms[t], truncs[t])
            ctx.eval_episodes(score[:T], terms[:T], truncs[:T], quota_d, slot_d, ep_return, ep_len, recorded, out_ret, out_len, remaining)

        graph, base = None, torch.zeros(1, dtype=torch.int64, device=dev)
        steps, rem = 0, int(remaining.item())
        while rem > 0:
            if steps >= max_steps:
                raise RuntimeError(f"evaluate(): environments {_unfinished(recorded.cpu().numpy(), quotas)} did not finish their "
                                   f"episodes within max_steps={max_steps} steps")
            T = min(S, max_steps - steps)
            if T == S and steps > 0 and graph is None and self.engine.use_graphs:
                # the chunk as one CUDA graph; the sampling counters baked into it are relative to a device-resident base
                graph = torch.cuda.CUDAGraph()
                torch.cuda.synchronize()
                ctx.set_draw_counter_base(base)
                try:
                    with torch.cuda.graph(graph):
                        chunk(S, lambda t: t)
                finally:
                    ctx.set_draw_counter_base(None)
            if T == S and graph is not None:
                base.fill_(gen["draws"])
                graph.replay()
            else:
                d0 = gen["draws"]
                chunk(T, lambda t: d0 + t)
            if not deterministic:
                gen["draws"] += T
            steps += T
            h_rem.copy_(remaining, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            rem = int(h_rem[0])
        return out_ret.cpu().numpy(), out_len.cpu().numpy().astype(np.int64)
