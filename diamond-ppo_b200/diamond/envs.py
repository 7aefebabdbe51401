"""Gymnasium-API environment shim.

The GPU image has no `gymnasium` (SURVEY.md §7 hard part 6).  The agents only need the small API
surface the reference touches (diamond/ppo.py:124-130, 163, 174-179, 291, 312): `spaces.Box/Discrete`,
an `Env` with reset/step, and a `SyncVectorEnv` with autoreset DISABLED whose `reset(options=
{"reset_mask": mask})` resets only the masked sub-envs.  If the real gymnasium is importable the
agents use it instead; these classes mirror its semantics.  CartPole-v1, Pendulum-v1, Acrobot-v1,
MountainCar-v0 and MountainCarContinuous-v0 follow the published Gymnasium dynamics; LunarLander needs
Box2D, so `SyntheticEnv(8, 4)` stands in for its shapes (obs 8, 4 actions).
"""
from __future__ import annotations

import math
from typing import Any, Callable

import numpy as np


class Space:
    pass


class Box(Space):
    def __init__(self, low=-np.inf, high=np.inf, shape=None, dtype=np.float32):
        if shape is None:
            shape = np.shape(low)
        self.shape = tuple(shape)
        self.low = np.broadcast_to(np.asarray(low, dtype=dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=dtype), self.shape).copy()
        self.dtype = np.dtype(dtype)


class Discrete(Space):
    def __init__(self, n: int):
        self.n = int(n)
        self.shape = ()
        self.dtype = np.dtype(np.int64)


class Env:
    observation_space: Space
    action_space: Space

    def reset(self, *, seed: int | None = None, options: dict | None = None):
        raise NotImplementedError

    def step(self, action):
        raise NotImplementedError

    def close(self):
        pass


class CartPoleEnv(Env):
    """CartPole-v1 dynamics (Barto, Sutton & Anderson 1983; Gymnasium classic_control), 500-step limit."""
    gravity, masscart, masspole, length, force_mag, tau = 9.8, 1.0, 0.1, 0.5, 10.0, 0.02
    theta_limit, x_limit, max_steps = 12 * 2 * math.pi / 360, 2.4, 500

    def __init__(self):
        high = np.array([self.x_limit * 2, np.inf, self.theta_limit * 2, np.inf], dtype=np.float32)
        self.observation_space = Box(-high, high, (4,))
        self.action_space = Discrete(2)
        self.rng = np.random.default_rng()
        self.state = np.zeros(4)
        self.t = 0

    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.state = self.rng.uniform(-0.05, 0.05, size=4)
        self.t = 0
        return self.state.astype(np.float32), {}

    def step(self, action):
        x, x_dot, th, th_dot = self.state
        force = self.force_mag if int(action) == 1 else -self.force_mag
        total_mass = self.masspole + self.masscart
        pml = self.masspole * self.length
        ct, st = math.cos(th), math.sin(th)
        temp = (force + pml * th_dot ** 2 * st) / total_mass
        th_acc = (self.gravity * st - ct * temp) / (self.length * (4.0 / 3.0 - self.masspole * ct ** 2 / total_mass))
        x_acc = temp - pml * th_acc * ct / total_mass
        self.state = np.array([x + self.tau * x_dot, x_dot + self.tau * x_acc, th + self.tau * th_dot, th_dot + self.tau * th_acc])
        self.t += 1
        terminated = bool(abs(self.state[0]) > self.x_limit or abs(self.state[2]) > self.theta_limit)
        truncated = bool(self.t >= self.max_steps and not terminated)
        return self.state.astype(np.float32), 1.0, terminated, truncated, {}


class PendulumEnv(Env):
    """Pendulum-v1 dynamics (Gymnasium classic_control), 200-step limit, torque in [-2, 2]."""
    max_speed, max_torque, dt, g, m, l, max_steps = 8.0, 2.0, 0.05, 10.0, 1.0, 1.0, 200

    def __init__(self):
        high = np.array([1.0, 1.0, self.max_speed], dtype=np.float32)
        self.observation_space = Box(-high, high, (3,))
        self.action_space = Box(-self.max_torque, self.max_torque, (1,))
        self.rng = np.random.default_rng()
        self.th, self.thdot, self.t = 0.0, 0.0, 0

    def _obs(self):
        return np.array([math.cos(self.th), math.sin(self.th), self.thdot], dtype=np.float32)

    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.th, self.thdot = self.rng.uniform(-math.pi, math.pi), self.rng.uniform(-1.0, 1.0)
        self.t = 0
        return self._obs(), {}

    def step(self, action):
        u = float(np.clip(np.asarray(action).reshape(-1)[0], -self.max_torque, self.max_torque))
        th_n = ((self.th + math.pi) % (2 * math.pi)) - math.pi
        cost = th_n ** 2 + 0.1 * self.thdot ** 2 + 0.001 * u ** 2
        self.thdot = float(np.clip(self.thdot + (3 * self.g / (2 * self.l) * math.sin(self.th) + 3.0 / (self.m * self.l ** 2) * u) * self.dt,
                                   -self.max_speed, self.max_speed))
        self.th += self.thdot * self.dt
        self.t += 1
        return self._obs(), -cost, False, self.t >= self.max_steps, {}


def _wrap(x, m, M):
    """Gymnasium's acrobot `wrap`: add or subtract the period until x lies in [m, M]."""
    diff = M - m
    while x > M:
        x = x - diff
    while x < m:
        x = x + diff
    return x


class AcrobotEnv(Env):
    """Acrobot-v1 (Sutton 1996; Gymnasium classic_control "book" dynamics): one RK4 step of dt 0.2, torque a - 1, 500-step limit."""
    dt, max_vel_1, max_vel_2, max_steps = 0.2, 4 * np.pi, 9 * np.pi, 500
    avail_torque = [-1.0, 0.0, +1]

    def __init__(self):
        high = np.array([1.0, 1.0, 1.0, 1.0, self.max_vel_1, self.max_vel_2], dtype=np.float32)
        self.observation_space = Box(-high, high, (6,))
        self.action_space = Discrete(3)
        self.rng = np.random.default_rng()
        self.state = np.zeros(4, dtype=np.float32)
        self.t = 0

    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.state = self.rng.uniform(-0.1, 0.1, size=4).astype(np.float32)
        self.t = 0
        return self._obs(), {}

    def _obs(self):
        s = self.state
        return np.array([np.cos(s[0]), np.sin(s[0]), np.cos(s[1]), np.sin(s[1]), s[2], s[3]], dtype=np.float32)

    @staticmethod
    def _dsdt(s_augmented):
        m1, m2, l1, lc1, lc2, I1, I2, g = 1.0, 1.0, 1.0, 0.5, 0.5, 1.0, 1.0, 9.8
        a = s_augmented[-1]
        theta1, theta2, dtheta1, dtheta2 = s_augmented[:-1]
        d1 = m1 * lc1 ** 2 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * np.cos(theta2)) + I1 + I2
        d2 = m2 * (lc2 ** 2 + l1 * lc2 * np.cos(theta2)) + I2
        phi2 = m2 * lc2 * g * np.cos(theta1 + theta2 - np.pi / 2.0)
        phi1 = (-m2 * l1 * lc2 * dtheta2 ** 2 * np.sin(theta2) - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * np.sin(theta2)
                + (m1 * lc1 + m2 * l1) * g * np.cos(theta1 - np.pi / 2) + phi2)
        ddtheta2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * dtheta1 ** 2 * np.sin(theta2) - phi2) / (m2 * lc2 ** 2 + I2 - d2 ** 2 / d1)
        ddtheta1 = -(d2 * ddtheta2 + phi1) / d1
        return dtheta1, dtheta2, ddtheta1, ddtheta2, 0.0

    def step(self, action):
        action = int(action)
        if not 0 <= action < 3:
            raise ValueError(f"Acrobot-v1 takes actions 0, 1, 2 (got {action})")
        torque = self.avail_torque[action]
        y0 = np.append(self.state, torque)             # float32 state after reset: promoted to float64 here
        dt = self.dt
        k1 = np.asarray(self._dsdt(y0))
        k2 = np.asarray(self._dsdt(y0 + dt / 2.0 * k1))
        k3 = np.asarray(self._dsdt(y0 + dt / 2.0 * k2))
        k4 = np.asarray(self._dsdt(y0 + dt * k3))
        ns = (y0 + dt / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4))[:4]
        ns[0] = _wrap(ns[0], -np.pi, np.pi)
        ns[1] = _wrap(ns[1], -np.pi, np.pi)
        ns[2] = min(max(ns[2], -self.max_vel_1), self.max_vel_1)
        ns[3] = min(max(ns[3], -self.max_vel_2), self.max_vel_2)
        self.state = ns
        self.t += 1
        terminated = bool(-np.cos(ns[0]) - np.cos(ns[1] + ns[0]) > 1.0)
        truncated = bool(self.t >= self.max_steps and not terminated)
        return self._obs(), -1.0 if not terminated else 0.0, terminated, truncated, {}


class MountainCarEnv(Env):
    """MountainCar-v0 (Moore 1990; Gymnasium classic_control): float64 state, force (a - 1) * 0.001, 200-step limit."""
    min_position, max_position, max_speed, goal_position, force, gravity, max_steps = -1.2, 0.6, 0.07, 0.5, 0.001, 0.0025, 200

    def __init__(self):
        self.observation_space = Box(np.array([self.min_position, -self.max_speed], dtype=np.float32),
                                     np.array([self.max_position, self.max_speed], dtype=np.float32), (2,))
        self.action_space = Discrete(3)
        self.rng = np.random.default_rng()
        self.state = np.zeros(2)
        self.t = 0

    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.state = np.array([self.rng.uniform(-0.6, -0.4), 0])
        self.t = 0
        return np.array(self.state, dtype=np.float32), {}

    def step(self, action):
        action = int(action)
        if not 0 <= action < 3:
            raise ValueError(f"MountainCar-v0 takes actions 0, 1, 2 (got {action})")
        position, velocity = self.state
        velocity += (action - 1) * self.force + math.cos(3 * position) * (-self.gravity)
        velocity = np.clip(velocity, -self.max_speed, self.max_speed)
        position += velocity
        position = np.clip(position, self.min_position, self.max_position)
        if position == self.min_position and velocity < 0:
            velocity = 0
        terminated = bool(position >= self.goal_position and velocity >= 0)
        self.state = (position, velocity)
        self.t += 1
        truncated = bool(self.t >= self.max_steps and not terminated)
        return np.array(self.state, dtype=np.float32), -1.0, terminated, truncated, {}


class MountainCarContinuousEnv(Env):
    """MountainCarContinuous-v0 (Gymnasium classic_control): float32 state, force min(max(a, -1), 1) * 0.0015, 999-step limit.
    Every step runs under NumPy 2's promotion rules (NEP 50): float32 arithmetic except math.cos and, for an action outside
    [-1, 1], the Python-float force term.  The reset state is float32 too, so the first step of an episode is no exception."""
    min_action, max_action, min_position, max_position, max_speed, goal_position, power, max_steps = \
        -1.0, 1.0, -1.2, 0.6, 0.07, 0.45, 0.0015, 999

    def __init__(self):
        self.observation_space = Box(np.array([self.min_position, -self.max_speed], dtype=np.float32),
                                     np.array([self.max_position, self.max_speed], dtype=np.float32), (2,))
        self.action_space = Box(self.min_action, self.max_action, (1,))
        self.rng = np.random.default_rng()
        self.state = np.zeros(2, dtype=np.float32)
        self.t = 0

    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.state = np.array([self.rng.uniform(-0.6, -0.4), 0], dtype=np.float32)
        self.t = 0
        return self.state.copy(), {}

    def step(self, action):
        action = np.asarray(action, dtype=np.float32).reshape(-1)
        position = self.state[0]
        velocity = self.state[1]
        force = min(max(action[0], self.min_action), self.max_action)
        velocity += force * self.power - 0.0025 * math.cos(3 * position)
        if velocity > self.max_speed:
            velocity = self.max_speed
        if velocity < -self.max_speed:
            velocity = -self.max_speed
        position += velocity
        if position > self.max_position:
            position = self.max_position
        if position < self.min_position:
            position = self.min_position
        if position == self.min_position and velocity < 0:
            velocity = 0
        terminated = bool(position >= self.goal_position and velocity >= 0)
        reward = 0
        if terminated:
            reward = 100.0
        reward -= math.pow(action[0], 2) * 0.1
        self.state = np.array([position, velocity], dtype=np.float32)
        self.t += 1
        truncated = bool(self.t >= self.max_steps and not terminated)
        return self.state.copy(), reward, terminated, truncated, {}


class SyntheticEnv(Env):
    """Shape-only stand-in (e.g. LunarLander-v3: obs 8, 4 actions): i.i.d. normal observations,
    reward depends on (obs, action), random terminations/truncations."""

    def __init__(self, obs_dim=8, n_actions=4, continuous=False, p_term=0.01, p_trunc=0.005):
        self.observation_space = Box(-np.inf, np.inf, (obs_dim,))
        self.action_space = Box(-1.0, 1.0, (n_actions,)) if continuous else Discrete(n_actions)
        self.continuous, self.p_term, self.p_trunc = continuous, p_term, p_trunc
        self.rng = np.random.default_rng()
        self.obs = np.zeros(obs_dim, np.float32)

    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.obs = self.rng.standard_normal(self.observation_space.shape).astype(np.float32)
        return self.obs, {}

    def step(self, action):
        a = float(np.sum(action)) if self.continuous else float(action)
        reward = float(self.obs[0]) * (1.0 if a > 0 else -1.0) * 0.1
        self.obs = self.rng.standard_normal(self.observation_space.shape).astype(np.float32)
        term = bool(self.rng.random() < self.p_term)
        trunc = bool((not term) and self.rng.random() < self.p_trunc)
        return self.obs, reward, term, trunc, {}


class SyncVectorEnv:
    """N sub-envs stepped serially; autoreset DISABLED (the caller resets done envs through
    reset(options={"reset_mask": mask}), so `step` returns the TRUE final observation, ppo.py:174-179)."""

    def __init__(self, env_fns: list[Callable[[], Env]], copy: bool = True, autoreset_mode: Any = "Disabled"):
        if str(autoreset_mode).lower().split(".")[-1] != "disabled":
            raise ValueError("this shim implements autoreset_mode='Disabled' only (what the agents use)")
        self.envs = [fn() for fn in env_fns]
        self.num_envs = len(self.envs)
        self.single_observation_space = self.envs[0].observation_space
        self.single_action_space = self.envs[0].action_space
        shape = self.single_observation_space.shape
        self._obs = np.zeros((self.num_envs,) + tuple(shape), dtype=np.float32)

    def reset(self, *, seed: int | None = None, options: dict | None = None):
        mask = None if options is None else options.get("reset_mask")
        for i, env in enumerate(self.envs):
            if mask is None or mask[i]:
                self._obs[i], _ = env.reset(seed=None if seed is None else seed + i)
        return self._obs.copy(), {}

    def step(self, actions):
        n = self.num_envs
        rewards = np.zeros(n, dtype=np.float64)
        terms = np.zeros(n, dtype=bool)
        truncs = np.zeros(n, dtype=bool)
        for i, env in enumerate(self.envs):
            self._obs[i], rewards[i], terms[i], truncs[i], _ = env.step(actions[i])
        return self._obs.copy(), rewards, terms, truncs, {}

    def close(self):
        for e in self.envs:
            e.close()


class BatchedSyntheticVectorEnv:
    """Vectorised synthetic env for large N (config S: 4096 envs would take seconds per step through
    N Python sub-envs).  Same vector API and autoreset-disabled semantics as SyncVectorEnv."""

    def __init__(self, num_envs, obs_dim=64, n_actions=4, continuous=False, p_term=0.01, p_trunc=0.01, seed=0):
        self.num_envs = num_envs
        self.single_observation_space = Box(-np.inf, np.inf, (obs_dim,))
        self.single_action_space = Box(-1.0, 1.0, (n_actions,)) if continuous else Discrete(n_actions)
        self.continuous, self.p_term, self.p_trunc = continuous, p_term, p_trunc
        self.rng = np.random.default_rng(seed)
        self._obs = np.zeros((num_envs, obs_dim), np.float32)

    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        mask = None if options is None else options.get("reset_mask")
        fresh = self.rng.standard_normal(self._obs.shape).astype(np.float32)
        self._obs = fresh if mask is None else np.where(np.asarray(mask)[:, None], fresh, self._obs)
        return self._obs.copy(), {}

    def step(self, actions):
        a = np.asarray(actions)
        a = a.reshape(self.num_envs, -1).sum(-1) if self.continuous else a
        rewards = (self._obs[:, 0] * np.where(a > 0, 1.0, -1.0) * 0.1).astype(np.float64)
        self._obs = self.rng.standard_normal(self._obs.shape).astype(np.float32)
        terms = self.rng.random(self.num_envs) < self.p_term
        truncs = (self.rng.random(self.num_envs) < self.p_trunc) & ~terms
        return self._obs.copy(), rewards, terms, truncs, {}

    def close(self):
        pass


class DeviceVectorEnv:
    """Vector environment that lives on the GPU (csrc/envs.cu: dppo_env_step / dppo_env_reset): CartPole-v1, Pendulum-v1,
    Acrobot-v1, MountainCar-v0, MountainCarContinuous-v0 (Gymnasium classic-control dynamics, float64 state; the continuous
    mountain car keeps Gymnasium's float32 state) and the synthetic shape stand-ins.  Same vector API and
    autoreset-DISABLED semantics as SyncVectorEnv, so any agent or user code can drive it through `step` / `reset` with host
    arrays; the default-network agents use `step_into`, which writes the step straight into the device rollout buffer and
    resets finished environments inside the same kernel (diamond/ppo.py:160-182 without a PCIe crossing).

    Use as `env_fn = DeviceVectorEnv.factory("CartPole-v1")` (an `env_fn.vectorized` factory taking num_envs).

    Normalisation (`normalize_observation`, `normalize_reward`): every environment keeps its own float64 statistics, exactly as one
    Gymnasium `NormalizeObservation(epsilon)` / `NormalizeReward(gamma, epsilon)` wrapper per sub-environment of a `SyncVectorEnv`
    would (optionally followed by a clip to +-`clip_observation` / +-`clip_reward`), inside the environment kernel: no host round
    trip and no extra launch per step.  Every emitted observation updates the statistics before it is normalised -- each step's
    final observation and each post-reset observation (in-kernel reset, `reset(options={"reset_mask": m})`, `reset(seed=...)`);
    the constructor's reset only brings the state up (it counts nothing and normalises with the initial statistics), as
    constructing a Gymnasium wrapper does not reset its environment.  The reward accumulator is cut by termination only, never by
    truncation or reset (Gymnasium's NormalizeReward).  `rewards` are the normalised rewards (what GAE consumes); `step()` returns
    the raw ones as `info["raw_rewards"]`, and agents pass a raw-reward row to `step_into` so episode returns stay raw.
    `update_running_mean = False` freezes both sets of statistics (it is read by the kernel from device memory, so replayed
    rollout graphs follow it).  The statistics are the tensors `obs_mean` [N, D], `obs_var` [N, D], `obs_count` [N] and
    `return_stats` [N, 4] (accumulator, mean, variance, count); include/dppo.h states the arithmetic."""

    device_resident = True
    _KINDS = {"CartPole-v1": (0, 4, 2, False), "Pendulum-v1": (1, 3, 1, True), "Acrobot-v1": (4, 6, 3, False),
              "MountainCar-v0": (5, 2, 3, False), "MountainCarContinuous-v0": (6, 2, 1, True)}

    def __init__(self, env_id: str, num_envs: int, seed: int = 0, device=None, obs_dim: int = 64, n_actions: int = 4,
                 continuous: bool = False, p_term: float = 0.01, p_trunc: float = 0.01, env_offset: int = 0,
                 normalize_observation: bool = False, normalize_reward: bool = False, gamma: float = 0.99, epsilon: float = 1e-8,
                 clip_observation: float | None = None, clip_reward: float | None = None):
        import torch
        from . import _native as N
        self._torch, self._N = torch, N
        if env_id in self._KINDS:
            kind, D, A, cont = self._KINDS[env_id]
        elif env_id in ("Synthetic", "LunarLander-v3"):                   # Box2D unavailable: shape stand-in
            D, A, cont = (8, 4, False) if env_id == "LunarLander-v3" else (int(obs_dim), int(n_actions), bool(continuous))
            kind = 3 if cont else 2
        else:
            raise KeyError(f"unknown device env id {env_id!r}; available: {sorted(self._KINDS) + ['LunarLander-v3', 'Synthetic']}")
        self.env_id, self.num_envs, self.continuous = env_id, int(num_envs), cont
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = N.get_context(self.device.index)
        if kind == 0:
            high = np.array([4.8, np.inf, 24 * math.pi / 360 * 2, np.inf], dtype=np.float32)
            self.single_observation_space, self.single_action_space = Box(-high, high, (4,)), Discrete(2)
        elif kind == 1:
            high = np.array([1.0, 1.0, 8.0], dtype=np.float32)
            self.single_observation_space, self.single_action_space = Box(-high, high, (3,)), Box(-2.0, 2.0, (1,))
        elif kind == 4:
            high = np.array([1.0, 1.0, 1.0, 1.0, 4 * np.pi, 9 * np.pi], dtype=np.float32)
            self.single_observation_space, self.single_action_space = Box(-high, high, (6,)), Discrete(3)
        elif kind in (5, 6):
            self.single_observation_space = Box(np.array([-1.2, -0.07], dtype=np.float32), np.array([0.6, 0.07], dtype=np.float32), (2,))
            self.single_action_space = Box(-1.0, 1.0, (1,)) if kind == 6 else Discrete(3)
        else:
            self.single_observation_space = Box(-np.inf, np.inf, (D,))
            self.single_action_space = Box(-1.0, 1.0, (A,)) if cont else Discrete(A)
        self.obs_dim, self.act_dim = D, A
        self._check_actions = kind in (4, 5)       # a host array may hold anything; the sampler's output is in range
        self.desc = N.EnvDesc(kind, self.num_envs, D, A, int(seed) & (2 ** 64 - 1), int(env_offset), float(p_term), float(p_trunc))
        for name, clip in (("clip_observation", clip_observation), ("clip_reward", clip_reward)):
            if clip is not None and not clip > 0:
                raise ValueError(f"{name} must be > 0 or None (got {clip})")
        self.normalize_observation, self.normalize_reward = bool(normalize_observation), bool(normalize_reward)
        if self.normalize_observation or self.normalize_reward:
            if not 0.0 <= gamma <= 1.0 or not epsilon > 0:
                raise ValueError(f"normalisation needs 0 <= gamma <= 1 and epsilon > 0 (got {gamma}, {epsilon})")
            self.desc.normalize = (N.ENV_NORMALIZE_OBS if self.normalize_observation else 0) | \
                (N.ENV_NORMALIZE_REWARD if self.normalize_reward else 0)
            self.desc.gamma, self.desc.epsilon = float(gamma), float(epsilon)
            self.desc.clip_observation, self.desc.clip_reward = float(clip_observation or 0.0), float(clip_reward or 0.0)
        if self.normalize_observation:                                  # as Gymnasium's NormalizeObservation
            self.single_observation_space = Box(-np.inf, np.inf, (D,))
        n, dev = self.num_envs, self.device
        self.state = torch.zeros(n, 4, dtype=torch.float64, device=dev)
        self.steps = torch.zeros(n, dtype=torch.int32, device=dev)
        self.episode = torch.zeros(n, dtype=torch.int64, device=dev)
        self.ep_return = torch.zeros(n, dtype=torch.float64, device=dev)
        self.cur_obs = torch.zeros(n, D, dtype=torch.float32, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        # normalisation statistics (Gymnasium's RunningMeanStd start: mean 0, var 1, count 1e-4) and the device freeze flag
        self.obs_mean = torch.zeros(n, D, **f64) if self.normalize_observation else None
        self.obs_var = torch.ones(n, D, **f64) if self.normalize_observation else None
        self.obs_count = torch.full((n,), 1e-4, **f64) if self.normalize_observation else None
        self.return_stats = torch.tensor([0.0, 0.0, 1.0, 1e-4], **f64).repeat(n, 1) if self.normalize_reward else None
        self._update = torch.ones(1, dtype=torch.int32, device=dev)
        self._update_running_mean = True
        ptr = lambda t: None if t is None else t.data_ptr()
        self._st = N.EnvState(self.state.data_ptr(), self.steps.data_ptr(), self.episode.data_ptr(), self.ep_return.data_ptr(),
                              self.cur_obs.data_ptr(), ptr(self.obs_mean), ptr(self.obs_var), ptr(self.obs_count),
                              ptr(self.return_stats), self._update.data_ptr())
        f = dict(dtype=torch.float32, device=dev)
        self._row = dict(next_obs=torch.empty(1, n, D, **f), rew=torch.empty(1, n, **f), term=torch.empty(1, n, **f),
                         trunc=torch.empty(1, n, **f), raw=torch.empty(1, n, **f) if self.normalize_reward else None)
        if self.desc.normalize:
            self._update.zero_()               # brings the state up without counting anything
        self.ctx.env_reset(self.desc, self._st, None)
        if self.desc.normalize:
            self._update.fill_(1)

    # the names of the tensors that hold the environments' state (checkpoints copy them)
    @property
    def state_tensors(self) -> tuple:
        names = ("state", "steps", "episode", "ep_return", "cur_obs")
        if self.normalize_observation:
            names += ("obs_mean", "obs_var", "obs_count")
        if self.normalize_reward:
            names += ("return_stats",)
        return names

    @property
    def update_running_mean(self) -> bool:
        """Whether steps and resets update the normalisation statistics (Gymnasium's property of the same name).  Setting it is
        stream-ordered: it takes effect for every launch (and graph replay) enqueued after it."""
        return self._update_running_mean

    @update_running_mean.setter
    def update_running_mean(self, value: bool) -> None:
        self._update_running_mean = bool(value)
        self._update.fill_(int(self._update_running_mean))

    def load_frozen_statistics(self, source: "DeviceVectorEnv") -> None:
        """Freezes this environment's normalisation statistics (update_running_mean = False) and gives environment i the
        statistics of `source`'s environment i mod source.num_envs: obs_mean / obs_var / obs_count and return_stats.  Evaluation
        environments take them from the training environments this way, which are only read."""
        torch = self._torch
        if (self.normalize_observation and not source.normalize_observation) or (self.normalize_reward and not source.normalize_reward):
            raise ValueError("load_frozen_statistics: the source environments do not keep every statistic this one normalises with")
        self.update_running_mean = False
        idx = torch.arange(self.num_envs, device=source.device) % source.num_envs
        names = (("obs_mean", "obs_var", "obs_count") if self.normalize_observation else ()) + \
            (("return_stats",) if self.normalize_reward else ())
        for name in names:
            getattr(self, name).copy_(getattr(source, name)[idx])

    @classmethod
    def factory(cls, env_id: str, **kwargs):
        def env_fn(num_envs):
            return cls(env_id, num_envs, **kwargs)
        env_fn.vectorized = True
        return env_fn

    def reset(self, *, seed: int | None = None, options: dict | None = None):
        torch = self._torch
        mask = None if options is None else options.get("reset_mask")
        if seed is not None:
            self.desc.seed = int(seed) & (2 ** 64 - 1)
            if mask is None:
                self.episode.zero_()
        m = None if mask is None else torch.as_tensor(np.asarray(mask, dtype=np.uint8) if not torch.is_tensor(mask) else mask).to(
            self.device, torch.uint8).contiguous()
        self.ctx.env_reset(self.desc, self._st, m)
        return self.cur_obs.cpu().numpy(), {}

    def _actions(self, actions):
        torch = self._torch
        a = actions if torch.is_tensor(actions) else torch.as_tensor(np.asarray(actions))
        if self.continuous:
            return a.to(self.device, torch.float32).reshape(self.num_envs, self.act_dim).contiguous()
        return a.to(self.device, torch.int64).reshape(self.num_envs).contiguous()

    def step(self, actions):
        """Gymnasium vector API with host arrays (autoreset disabled: the caller resets through reset(options=...))."""
        r = self._row
        a = self._actions(actions)
        if self._check_actions and bool(((a < 0) | (a >= self.act_dim)).any()):
            raise ValueError(f"{self.env_id} takes actions 0 .. {self.act_dim - 1}; got {a.min().item()} .. {a.max().item()}")
        self.ctx.env_step(self.desc, self._st, a, 0, False, None, r["next_obs"], None, r["rew"], r["term"], r["trunc"],
                          raw_rewards=r["raw"])
        info = {} if r["raw"] is None else {"raw_rewards": r["raw"][0].double().cpu().numpy()}
        return (r["next_obs"][0].cpu().numpy(), r["rew"][0].double().cpu().numpy(), r["term"][0].bool().cpu().numpy(),
                r["trunc"][0].bool().cpu().numpy(), info)

    def step_into(self, buf, t: int, actions) -> None:
        """Fused rollout step: row t of the device rollout buffer (obs, next_obs, actions, rewards, terminations, truncations,
        and raw_rewards when the buffer has that attribute) is written by the kernel, finished environments are reset, `cur_obs`
        becomes the next step's observations."""
        self.ctx.env_step(self.desc, self._st, self._actions(actions), t, True, buf.obs, buf.next_obs, buf.actions, buf.rewards,
                          buf.terminations, buf.truncations, raw_rewards=getattr(buf, "raw_rewards", None))
        buf.filled = max(buf.filled, t + 1)

    def close(self):
        pass


_REGISTRY = {"CartPole-v1": CartPoleEnv, "Pendulum-v1": PendulumEnv, "Acrobot-v1": AcrobotEnv, "MountainCar-v0": MountainCarEnv,
             "MountainCarContinuous-v0": MountainCarContinuousEnv,
             "LunarLander-v3": lambda: SyntheticEnv(8, 4)}       # Box2D unavailable: shape stand-in


def make(env_id: str, **kwargs) -> Env:
    """gym.make for the ids BASELINE.json's configs name."""
    if env_id not in _REGISTRY:
        raise KeyError(f"unknown env id {env_id!r}; available: {sorted(_REGISTRY)}")
    return _REGISTRY[env_id](**kwargs) if kwargs else _REGISTRY[env_id]()


class _Namespace:
    pass


# `import diamond.envs as gym` then gym.spaces.Box / gym.vector.SyncVectorEnv / gym.make work
spaces = _Namespace()
spaces.Space, spaces.Box, spaces.Discrete = Space, Box, Discrete
vector = _Namespace()
vector.SyncVectorEnv = SyncVectorEnv
