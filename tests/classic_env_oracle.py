"""TEST INFRASTRUCTURE ONLY — CPU restatement of the Acrobot-v1, MountainCar-v0 and MountainCarContinuous-v0 dynamics that the
device environments (csrc/envs.cu kinds 4, 5, 6) implement; the CartPole-v1 / Pendulum-v1 restatement is oracle/env_oracle.py.
Not part of the product: only tests/ import this module.  Same signature as oracle/env_oracle.py's `cartpole_step`:
(state [N, 4+] float64, actions, steps taken so far) -> next_state, obs f32, reward, terminated, truncated.

The dynamics are third-party Gymnasium code (`gymnasium>=1.0.0`, not installed here), restated from its classic-control sources:

* Acrobot-v1 — gymnasium/envs/classic_control/acrobot.py `AcrobotEnv.step` / `_dsdt` / `rk4` / `wrap` / `bound` (Sutton 1996,
  "book" dynamics): m1 = m2 = l1 = 1, lc1 = lc2 = 0.5, I1 = I2 = 1, g 9.8, torque a - 1 (no noise); one classical RK4 step over
  [0, 0.2]; theta1, theta2 wrapped into [-pi, pi] by adding / subtracting 2 pi, speeds bounded to 4 pi / 9 pi; terminated when
  -cos th1 - cos(th1 + th2) > 1; reward -1, 0 on the terminating step; TimeLimit 500; reset U(-0.1, 0.1)^4 rounded to float32
  (`.astype(np.float32)`), promoted to float64 by the first step's `np.append`; obs (cos th1, sin th1, cos th2, sin th2, dth1, dth2).
* MountainCar-v0 — gymnasium/envs/classic_control/mountain_car.py `MountainCarEnv.step` (Moore 1990): float64;
  v += (a - 1) 0.001 + cos(3 p) (-0.0025), v clipped to +-0.07, p += v clipped to [-1.2, 0.6], v = 0 at the left wall when v < 0;
  terminated when p >= 0.5 and v >= 0; reward -1; TimeLimit 200; reset p ~ U(-0.6, -0.4), v = 0.
* MountainCarContinuous-v0 — gymnasium/envs/classic_control/continuous_mountain_car.py `Continuous_MountainCarEnv.step`: the
  state is float32 and NumPy 2 (NEP 50) runs every operation and comparison of the step in float32, Python constants rounded to
  float32 -- except `math.cos(3 * position)` (double of the float32 product) and, for an action outside [-1, 1], the force term
  `+-1.0 * 0.0015 - 0.0025 cos` (the clamp returns a Python float: double, rounded once into the velocity update); speed clip
  +-0.07, position clip [-1.2, 0.6] with the left-wall rule; terminated when p >= 0.45 and v >= 0; reward (100 if terminated)
  - 0.1 a^2 in double on the unclipped action; TimeLimit 999; reset p = float32 of U(-0.6, -0.4), v = 0.
Time limits follow the repository's convention, truncated = steps >= limit and not terminated, which gives the same GAE inputs
and `done` as Gymnasium's TimeLimit.  The project is tested under NumPy 2.x; the promotion notes above assume it.

parity unpinned by golden vectors of gymnasium itself (absent); pinned against the independent per-env host implementation in
diamond/envs.py (tests/test_classic_envs.py) and against hand-computed single steps."""
import math

import numpy as np


def _wrap(x, m, M):
    diff = M - m
    while np.any(x > M):
        x = np.where(x > M, x - diff, x)
    while np.any(x < m):
        x = np.where(x < m, x + diff, x)
    return x


def _acrobot_dsdt(y, torque):
    m1, m2, l1, lc1, lc2, I1, I2, g = 1.0, 1.0, 1.0, 0.5, 0.5, 1.0, 1.0, 9.8
    th1, th2, dth1, dth2 = y
    d1 = m1 * lc1 ** 2 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * np.cos(th2)) + I1 + I2
    d2 = m2 * (lc2 ** 2 + l1 * lc2 * np.cos(th2)) + I2
    phi2 = m2 * lc2 * g * np.cos(th1 + th2 - np.pi / 2.0)
    phi1 = (-m2 * l1 * lc2 * dth2 ** 2 * np.sin(th2) - 2 * m2 * l1 * lc2 * dth2 * dth1 * np.sin(th2)
            + (m1 * lc1 + m2 * l1) * g * np.cos(th1 - np.pi / 2) + phi2)
    ddth2 = (torque + d2 / d1 * phi1 - m2 * l1 * lc2 * dth1 ** 2 * np.sin(th2) - phi2) / (m2 * lc2 ** 2 + I2 - d2 ** 2 / d1)
    return [dth1, dth2, -(d2 * ddth2 + phi1) / d1, ddth2]


def acrobot_step(state: np.ndarray, actions: np.ndarray, steps: np.ndarray):
    """state [N,4] float64 (th1, th2, dth1, dth2), actions [N] int in {0, 1, 2} -> next_state, obs f32 [N,6], reward, terminated,
    truncated."""
    y0 = [state[:, i].astype(np.float64) for i in range(4)]
    torque = np.asarray(actions).astype(np.float64) - 1.0
    dt = 0.2
    k1 = _acrobot_dsdt(y0, torque)
    k2 = _acrobot_dsdt([y + dt / 2.0 * k for y, k in zip(y0, k1)], torque)
    k3 = _acrobot_dsdt([y + dt / 2.0 * k for y, k in zip(y0, k2)], torque)
    k4 = _acrobot_dsdt([y + dt * k for y, k in zip(y0, k3)], torque)
    ns = [y + dt / 6.0 * (a + 2 * b + 2 * c + d) for y, a, b, c, d in zip(y0, k1, k2, k3, k4)]
    ns[0], ns[1] = _wrap(ns[0], -np.pi, np.pi), _wrap(ns[1], -np.pi, np.pi)
    ns[2] = np.minimum(np.maximum(ns[2], -4 * np.pi), 4 * np.pi)
    ns[3] = np.minimum(np.maximum(ns[3], -9 * np.pi), 9 * np.pi)
    nxt = np.stack(ns, axis=1)
    terminated = -np.cos(ns[0]) - np.cos(ns[1] + ns[0]) > 1.0
    obs = np.stack([np.cos(ns[0]), np.sin(ns[0]), np.cos(ns[1]), np.sin(ns[1]), ns[2], ns[3]], axis=1).astype(np.float32)
    truncated = ((np.asarray(steps) + 1) >= 500) & ~terminated
    return nxt, obs, np.where(terminated, 0.0, -1.0), terminated, truncated


def _math_cos(x):
    """math.cos element by element (libm double), as Gymnasium's mountain cars call it."""
    return np.array([math.cos(v) for v in np.asarray(x, dtype=np.float64).reshape(-1)], dtype=np.float64)


def mountain_car_step(state: np.ndarray, actions: np.ndarray, steps: np.ndarray):
    """state [N,2+] float64 (position, velocity), actions [N] int in {0, 1, 2} -> next_state [N,2], obs f32 [N,2], reward,
    terminated, truncated."""
    p, v = state[:, 0].astype(np.float64), state[:, 1].astype(np.float64)
    v = v + ((np.asarray(actions).astype(np.int64) - 1) * 0.001 + _math_cos(3 * p) * (-0.0025))
    v = np.clip(v, -0.07, 0.07)
    p = np.clip(p + v, -1.2, 0.6)
    v = np.where((p == -1.2) & (v < 0), 0.0, v)
    terminated = (p >= 0.5) & (v >= 0)
    nxt = np.stack([p, v], axis=1)
    return nxt, nxt.astype(np.float32), -np.ones(len(p)), terminated, ((np.asarray(steps) + 1) >= 200) & ~terminated


def mountain_car_continuous_step(state: np.ndarray, actions: np.ndarray, steps: np.ndarray):
    """state [N,2+] float32-representable (position, velocity), actions [N,1] float -> next_state [N,2] (float32 values held in
    float64), obs f32 [N,2], reward, terminated, truncated."""
    f32 = np.float32
    p, v = state[:, 0].astype(f32), state[:, 1].astype(f32)
    a = np.asarray(actions, dtype=f32).reshape(len(p), -1)[:, 0]
    gc = 0.0025 * _math_cos(f32(3) * p)                                  # Python float (double)
    in_range = ~((a < -1.0) | (a > 1.0))
    dv = np.where(in_range, a * f32(0.0015) - gc.astype(f32),            # float32 multiply and subtract
                  (np.where(a > 1.0, 1.0, -1.0) * 0.0015 - gc).astype(f32))  # double, rounded once
    v = v + dv
    v = np.where(v > f32(0.07), f32(0.07), v)
    v = np.where(v < f32(-0.07), f32(-0.07), v)
    p = p + v
    p = np.where(p > f32(0.6), f32(0.6), p)
    p = np.where(p < f32(-1.2), f32(-1.2), p)
    v = np.where((p == f32(-1.2)) & (v < 0), f32(0), v)
    terminated = (p >= f32(0.45)) & (v >= 0)
    reward = np.where(terminated, 100.0, 0.0) - a.astype(np.float64) ** 2 * 0.1
    obs = np.stack([p, v], axis=1)
    return obs.astype(np.float64), obs, reward, terminated, ((np.asarray(steps) + 1) >= 999) & ~terminated
