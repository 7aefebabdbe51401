"""CPU: tests/classic_env_oracle.py's Acrobot-v1 / MountainCar-v0 / MountainCarContinuous-v0 steps against the independent
per-env host classes in diamond/envs.py, over states drawn across and beyond the reachable range, plus hand-computed steps."""
import math
import os
import sys

import numpy as np
import pytest

from diamond import envs

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import classic_env_oracle as EO  # noqa: E402

TWO_PI = 2 * np.pi


def _one(step_fn, state, action, t0):
    nxt, obs, r, term, trunc = step_fn(np.asarray(state, dtype=np.float64)[None], np.asarray(action)[None], np.array([t0]))
    return nxt[0], obs[0], float(r[0]), bool(term[0]), bool(trunc[0])


def _check(env, ref, obs, rew, term, trunc, state, exact_state):
    nxt, robs, rr, rterm, rtrunc = ref
    if exact_state:
        np.testing.assert_array_equal(nxt, state)
    else:
        np.testing.assert_allclose(nxt, state, rtol=1e-13, atol=1e-15)
    np.testing.assert_array_equal(robs, obs)
    assert (rterm, rtrunc, rr) == (term, trunc, rew)


def test_acrobot_oracle_matches_host_class():
    rng = np.random.default_rng(0)
    seen = dict(term=0, trunc=0, wrap_twice=0, bound=0)
    states = []
    for i in range(400):
        s = np.concatenate([rng.uniform(-TWO_PI, TWO_PI, 2), rng.uniform(-1.5, 1.5, 2) * np.array([4 * np.pi, 9 * np.pi])])
        if i % 8 == 0:                                     # close to the goal: termination, and wrap from just below +-2 pi
            s[:2] = [np.pi * rng.uniform(0.7, 1.3), rng.uniform(-0.5, 0.5)]
        if i % 8 == 1:
            s[0], s[2] = np.sign(s[2]) * rng.uniform(1.8, 2.0) * np.pi, np.sign(s[2]) * rng.uniform(4.0, 6.0) * np.pi
        states.append(s)
    for i, s0 in enumerate(states):
        e = envs.AcrobotEnv()
        e.state = s0.copy()
        e.t = int(rng.integers(0, 500)) if i % 5 else 499        # every fifth step is the last one of the time limit
        t0, a = e.t, int(rng.integers(0, 3))
        obs, rew, term, trunc, _ = e.step(a)
        _check(e, _one(EO.acrobot_step, s0, a, t0), obs, rew, term, trunc, e.state, False)
        assert np.all(np.abs(e.state[:2]) <= np.pi)
        assert abs(e.state[2]) <= 4 * np.pi and abs(e.state[3]) <= 9 * np.pi
        seen["term"] += term
        seen["trunc"] += trunc
        seen["wrap_twice"] += bool(np.abs(s0[0] + 0.2 * s0[2]) > 3 * np.pi)   # the first angle leaves [-3 pi, 3 pi] during the step
        seen["bound"] += bool(abs(e.state[2]) == 4 * np.pi or abs(e.state[3]) == 9 * np.pi)
    assert all(v > 0 for v in seen.values()), seen


def test_mountain_car_oracle_matches_host_class():
    rng = np.random.default_rng(1)
    seen = dict(term=0, trunc=0, wall=0, clip_v=0, right=0)
    for i in range(400):
        e = envs.MountainCarEnv()
        k = i % 5
        if k == 0:                                         # at and beyond the left wall, moving left
            s0 = np.array([rng.choice([-1.2, -1.25, -1.19]), -rng.uniform(0.0, 0.1)])
        elif k == 1:                                       # at the goal thresholds
            s0 = np.array([rng.choice([0.5, 0.499, 0.4995]), rng.choice([0.0, 0.001, -1e-4])])
        elif k == 2:                                       # past the speed bound, at and beyond the right wall
            s0 = np.array([rng.uniform(0.55, 0.7), rng.choice([-1, 1]) * rng.uniform(0.06, 0.1)])
        else:
            s0 = np.array([rng.uniform(-1.3, 0.7), rng.uniform(-0.08, 0.08)])
        e.state = (float(s0[0]), float(s0[1]))
        e.t = int(rng.integers(0, 200)) if i % 7 else 199
        t0, a = e.t, int(rng.integers(0, 3))
        obs, rew, term, trunc, _ = e.step(a)
        state = np.array(e.state, dtype=np.float64)
        _check(e, _one(EO.mountain_car_step, s0, a, t0), obs, rew, term, trunc, state, False)
        seen["term"] += term
        seen["trunc"] += trunc
        seen["wall"] += bool(state[0] == -1.2 and state[1] == 0.0)
        seen["clip_v"] += bool(abs(state[1]) == 0.07)
        seen["right"] += bool(state[0] == 0.6)
    assert all(v > 0 for v in seen.values()), seen


def test_mountain_car_continuous_oracle_matches_host_class_bit_exactly():
    rng = np.random.default_rng(2)
    f32 = np.float32
    seen = dict(term=0, trunc=0, wall=0, clip_v=0, right=0, out_of_range=0, unit=0)
    for i in range(600):
        e = envs.MountainCarContinuousEnv()
        k = i % 5
        if k == 0:
            s0 = [rng.choice([-1.2, -1.25, -1.19]), -rng.uniform(0.0, 0.1)]
        elif k == 1:
            s0 = [rng.choice([0.45, 0.449, 0.4499]), rng.choice([0.0, 0.001, -1e-4])]
        elif k == 2:
            s0 = [rng.uniform(0.55, 0.7), rng.choice([-1, 1]) * rng.uniform(0.06, 0.1)]
        else:
            s0 = [rng.uniform(-1.3, 0.7), rng.uniform(-0.08, 0.08)]
        s0 = np.array(s0, dtype=f32)                       # Gymnasium's float32 state
        a = np.array([rng.choice([1.0, -1.0]) if i % 11 == 0 else rng.uniform(-3, 3)], dtype=f32)
        e.state = s0.copy()
        e.t = int(rng.integers(0, 999)) if i % 7 else 998
        obs, rew, term, trunc, _ = e.step(a)
        _check(e, _one(EO.mountain_car_continuous_step, s0, a[None], e.t - 1), obs, rew, term, trunc, e.state.astype(np.float64), True)
        assert e.state.dtype == np.float32
        seen["term"] += term
        seen["trunc"] += trunc
        seen["wall"] += bool(e.state[0] == f32(-1.2) and e.state[1] == 0)
        seen["clip_v"] += bool(abs(e.state[1]) == f32(0.07))
        seen["right"] += bool(e.state[0] == f32(0.6))
        seen["out_of_range"] += bool(abs(a[0]) > 1)
        seen["unit"] += bool(abs(a[0]) == 1)
    assert all(v > 0 for v in seen.values()), seen


def test_mountain_car_hand_computed_step():
    """(-0.5, 0), action 2: v = 0 + (1 * 0.001 + cos(-1.5) * -0.0025) with cos(1.5) = 0.0707372016677029..., p = -0.5 + v."""
    nxt, obs, r, term, trunc = _one(EO.mountain_car_step, [-0.5, 0.0], 2, 0)
    v = 0.001 - 0.0025 * 0.0707372016677029100881
    np.testing.assert_allclose(nxt, [-0.5 + v, v], rtol=1e-15)
    np.testing.assert_allclose(v, 8.23156995830742725e-4, rtol=1e-15)
    assert r == -1.0 and not term and not trunc
    np.testing.assert_array_equal(obs, np.array([-0.5 + v, v], dtype=np.float32))


def test_mountain_car_continuous_hand_computed_step():
    """(-0.5, 0), action 0.5, every operation of the step in float32 except the double cos and 0.0025 * cos:
    3 * p = -1.5 (float32, exact); c = cos(-1.5) in double; force * power = f32(0.5) * f32(0.0015) rounded to float32;
    dv = that - f32(0.0025 * c), rounded to float32; v = f32(0) + dv; p = f32(-0.5) + v; reward = -0.1 * 0.25 in double."""
    f32 = np.float32
    nxt, obs, r, term, trunc = _one(EO.mountain_car_continuous_step, [-0.5, 0.0], [0.5], 0)
    c = math.cos(-1.5)
    fp = f32(f32(0.5) * f32(0.0015))                     # f32(0.0015) = 0.001500000013038516..., halved exactly
    assert float(fp) == 0.5 * 0.0015000000130385160446
    g = f32(0.0025 * c)                                   # 1.76843004169257e-4 rounded to float32
    dv = f32(fp - g)
    v = f32(f32(0.0) + dv)
    p = f32(f32(-0.5) + v)
    np.testing.assert_array_equal(nxt, np.array([p, v], dtype=np.float64))
    np.testing.assert_array_equal(obs, np.array([p, v], dtype=f32))
    assert abs(float(v) - (0.5 * 0.0015 - 0.0025 * c)) < 1e-10       # the intended quantity, up to float32 rounding
    assert r == -(0.25 * 0.1) and not term and not trunc


@pytest.mark.parametrize("env_id", ["Acrobot-v1", "MountainCar-v0", "MountainCarContinuous-v0"])
def test_host_reset_draws_and_time_limits(env_id):
    e = envs.make(env_id)
    for seed in range(50):
        obs, _ = e.reset(seed=seed)
        assert obs.dtype == np.float32 and obs.shape == e.observation_space.shape
        s = np.asarray(e.state)
        if env_id == "Acrobot-v1":
            assert s.dtype == np.float32 and np.all(np.abs(s) <= 0.1)
            np.testing.assert_allclose(obs, [np.cos(s[0]), np.sin(s[0]), np.cos(s[1]), np.sin(s[1]), s[2], s[3]], atol=1e-7)
        else:
            assert -0.6 <= s[0] <= -0.4 and s[1] == 0
            assert np.array_equal(obs, s.astype(np.float32))
            assert (s.dtype == np.float32) == (env_id == "MountainCarContinuous-v0")
    limit, action = {"Acrobot-v1": (500, 1), "MountainCar-v0": (200, 1), "MountainCarContinuous-v0": (999, np.zeros(1, np.float32))}[env_id]
    e.reset(seed=0)
    for t in range(limit):
        _, _, term, trunc, _ = e.step(action)
        assert not term and trunc == (t == limit - 1)


@pytest.mark.parametrize("env_id", ["Acrobot-v1", "MountainCar-v0"])
def test_host_discrete_envs_refuse_actions_outside_range(env_id):
    e = envs.make(env_id)
    e.reset(seed=0)
    for bad in (-1, 3):
        with pytest.raises(ValueError):
            e.step(bad)


@pytest.mark.parametrize("env_id", ["Acrobot-v1", "MountainCar-v0", "MountainCarContinuous-v0"])
def test_sync_vector_env_runs_new_ids(env_id):
    vec = envs.vector.SyncVectorEnv([lambda: envs.make(env_id) for _ in range(4)])
    obs, _ = vec.reset(seed=3)
    cont = isinstance(vec.single_action_space, envs.Box)
    rng = np.random.default_rng(0)
    for _ in range(20):
        act = rng.uniform(-1, 1, (4, 1)).astype(np.float32) if cont else rng.integers(0, 3, 4)
        obs, rew, term, trunc, _ = vec.step(act)
        assert obs.shape == (4,) + vec.single_observation_space.shape and np.all(np.isfinite(obs))
        if np.any(term | trunc):
            vec.reset(options={"reset_mask": term | trunc})
