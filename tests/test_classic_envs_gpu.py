"""GPU: the Acrobot-v1 / MountainCar-v0 / MountainCarContinuous-v0 device environments (csrc/envs.cu kinds 4-6) against
tests/classic_env_oracle.py, and every agent path that drives them."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

# PPO on device Acrobot-v1 with the default hyper-parameters, 64 envs x 128 steps.  Mean length of the last 100 episodes measured on
# one B200 (1000 W power limit): seed 1: 429 / 330 / 199 / 131 / 105 after 10 / 20 / 30 / 40 / 60 rollouts; seed 2: 493 / 473 / 453 /
# 446 / 165 -- a random policy mostly runs into the 500-step cap.  60 rollouts and a bound of 300 leave room for a slower seed.
ACROBOT_ROLLOUTS, ACROBOT_MAX_MEAN_LENGTH = 60, 300.0
IDS = ["Acrobot-v1", "MountainCar-v0", "MountainCarContinuous-v0"]
LIMIT = {"Acrobot-v1": 500, "MountainCar-v0": 200, "MountainCarContinuous-v0": 999}
# (agent, env id) pairs: every agent that takes the id's action space
AGENT_PAIRS = [("PPO", "Acrobot-v1"), ("PPO", "MountainCar-v0"), ("ContinuousPPO", "MountainCarContinuous-v0"), ("RecurrentPPO", "Acrobot-v1")]


def _oracle(env_id):
    import classic_env_oracle as EO
    return {"Acrobot-v1": EO.acrobot_step, "MountainCar-v0": EO.mountain_car_step,
            "MountainCarContinuous-v0": EO.mountain_car_continuous_step}[env_id]


def _random_states(env_id, rng, n):
    """States across and beyond the reachable range: several wraps, speeds past their bounds, both walls, the goal thresholds."""
    if env_id == "Acrobot-v1":
        s = np.concatenate([rng.uniform(-2, 2, (n, 2)) * np.pi, rng.uniform(-1.5, 1.5, (n, 2)) * np.array([4 * np.pi, 9 * np.pi])], 1)
        near_goal = rng.random(n) < 0.3
        s[near_goal, 0] = np.pi * rng.uniform(0.7, 1.3, near_goal.sum())
        s[near_goal, 1] = rng.uniform(-0.5, 0.5, near_goal.sum())
        return s
    goal = 0.5 if env_id == "MountainCar-v0" else 0.45
    p = rng.uniform(-1.3, 0.7, n)
    v = rng.uniform(-0.09, 0.09, n)
    k = rng.integers(0, 3, n)
    p[k == 0] = rng.choice([-1.2, -1.21, -1.19], (k == 0).sum())
    v[k == 0] = -np.abs(v[k == 0])
    p[k == 1] = goal - rng.choice([0.0, 1e-3, 1e-4], (k == 1).sum())
    v[k == 1] = rng.choice([0.0, 1e-3, -1e-4], (k == 1).sum())
    s = np.stack([p, v], 1)
    return s.astype(np.float32).astype(np.float64) if env_id == "MountainCarContinuous-v0" else s


def _actions(env_id, rng, n):
    if env_id == "MountainCarContinuous-v0":
        a = rng.uniform(-3, 3, (n, 1)).astype(np.float32)
        a[rng.random(n) < 0.1, 0] = rng.choice([-1.0, 1.0])
        return a
    return rng.integers(0, 3, n)


def _float64_tolerance(step_fn, state, actions, steps, ref_next, rng):
    """1e-12 (absolute and relative), widened where the step itself amplifies rounding: 32 times the oracle's own change when its
    input moves by one ulp (largest over four random sign patterns).  One Acrobot RK4 step from a fast state (|theta2_dot| near
    9 pi) turns a one-ulp change of the input into up to ~4e-10 of the output, so CUDA's cos / sin and fused multiply-adds, each
    within an ulp or two of NumPy's, cannot agree with the oracle to 1e-12 there; elsewhere the bound stays at 1e-12."""
    sens = np.zeros_like(ref_next)
    for _ in range(4):
        pert = state * (1 + np.finfo(np.float64).eps * rng.choice([-1.0, 1.0], state.shape))
        d = np.abs(step_fn(pert, actions, steps)[0] - ref_next)
        sens = np.maximum(sens, np.minimum(d, np.abs(d - 2 * np.pi)))     # a wrapped angle may move by 2 pi
    return 1e-12 * (1 + np.abs(ref_next)) + 32 * sens


@pytest.mark.parametrize("env_id", IDS)
def test_device_env_steps_match_oracle(env_id):
    """600 vector steps of 96 environments with random actions, masked resets, and random states / step counts written into the
    environment before every fifth step: flags bit-exact, float64 state to 1e-12 except where the step amplifies rounding
    (_float64_tolerance), MountainCarContinuous's float32 state within one float32 ulp, observations to 1e-6, rewards equal to
    the oracle's rounded to float32."""
    from diamond.envs import DeviceVectorEnv
    N_ = 96
    env = DeviceVectorEnv(env_id, N_, seed=5)
    step_fn = _oracle(env_id)
    rng = np.random.default_rng(1)
    env.reset(seed=5)
    seen = dict(term=0, trunc=0, reset=0, edge=0)
    cont = env_id == "MountainCarContinuous-v0"
    ulp_off = 0
    sens_rng = np.random.default_rng(7)
    for it in range(600):
        if it % 5 == 0:
            idx = torch.as_tensor(np.flatnonzero(rng.random(N_) < 0.4), device=env.device)
            st = torch.as_tensor(_random_states(env_id, rng, len(idx)), device=env.device)
            env.state[idx, :st.shape[1]] = st
            if it % 10 == 0:                                         # the last steps before the time limit
                env.steps[idx] = torch.as_tensor(rng.integers(LIMIT[env_id] - 3, LIMIT[env_id], len(idx)), dtype=torch.int32,
                                                 device=env.device)
        state = env.state.cpu().numpy().copy()
        steps = env.steps.cpu().numpy().copy()
        actions = _actions(env_id, rng, N_)
        nobs, rew, term, trunc, _ = env.step(actions)
        ref_next, ref_obs, ref_rew, ref_term, ref_trunc = step_fn(state, actions, steps)
        got = env.state.cpu().numpy()[:, :ref_next.shape[1]]
        np.testing.assert_array_equal(term, ref_term)
        np.testing.assert_array_equal(trunc, ref_trunc)
        if cont:
            # exact except where CUDA's double cos and libm's differ by an ulp across a float32 rounding boundary
            ref32 = ref_next.astype(np.float32)
            assert np.array_equal(got, got.astype(np.float32).astype(np.float64))
            assert np.all(np.abs(got - ref_next) <= np.spacing(np.abs(ref32)).astype(np.float64))
            ulp_off += int((got != ref_next).sum())
        else:
            err = np.abs(got - ref_next)
            tol = _float64_tolerance(step_fn, state, actions, steps, ref_next, sens_rng)
            assert np.all(err <= tol), (it, np.argwhere(err > tol), err[err > tol], tol[err > tol])
        np.testing.assert_allclose(nobs, ref_obs, rtol=0, atol=1e-6)
        np.testing.assert_array_equal(rew, ref_rew.astype(np.float32).astype(np.float64))
        if env_id == "Acrobot-v1":
            seen["edge"] += int((np.abs(state[:, 0] + 0.2 * state[:, 2]) > 3 * np.pi).sum())     # wrap runs more than once
        else:
            seen["edge"] += int(((got[:, 0] == np.float32(-1.2) if cont else got[:, 0] == -1.2) & (got[:, 1] == 0)).sum())   # wall rule
        seen["term"] += int(term.sum())
        seen["trunc"] += int(trunc.sum())
        dones = term | trunc
        if dones.any():
            seen["reset"] += 1
            before = env.state.cpu().numpy().copy()
            obs, _ = env.reset(options={"reset_mask": dones})
            after = env.state.cpu().numpy()
            assert np.array_equal(after[~dones], before[~dones])
            assert np.all(env.steps.cpu().numpy()[dones] == 0)
            assert np.array_equal(obs[~dones], nobs[~dones])
    assert all(v > 0 for v in seen.values()), seen
    assert ulp_off <= 4, ulp_off


@pytest.mark.parametrize("env_id", IDS)
def test_device_reset_draws_are_in_range_and_keyed_by_seed_and_global_env_id(env_id):
    from diamond.envs import DeviceVectorEnv
    a = DeviceVectorEnv(env_id, 32, seed=9)
    b = DeviceVectorEnv(env_id, 16, seed=9, env_offset=16)          # the second shard of a 32-env run
    c = DeviceVectorEnv(env_id, 32, seed=10)
    assert torch.equal(a.state[16:], b.state) and torch.equal(a.cur_obs[16:], b.cur_obs)
    assert not torch.equal(a.state, c.state)
    big = DeviceVectorEnv(env_id, 4096, seed=1)
    s = big.state.cpu().numpy()
    obs = big.cur_obs.cpu().numpy()
    if env_id == "Acrobot-v1":
        assert np.all(np.abs(s) <= float(np.float32(0.1))) and np.array_equal(s, s.astype(np.float32).astype(np.float64))
        assert s.std(0).min() > 0.05                                 # spread over the whole interval, all four coordinates
        ref = np.stack([np.cos(s[:, 0]), np.sin(s[:, 0]), np.cos(s[:, 1]), np.sin(s[:, 1]), s[:, 2], s[:, 3]], 1).astype(np.float32)
        np.testing.assert_allclose(obs, ref, atol=1e-7)
    else:
        lo, hi = (float(np.float32(-0.6)), float(np.float32(-0.4))) if env_id == "MountainCarContinuous-v0" else (-0.6, -0.4)
        assert np.all((s[:, 0] >= lo) & (s[:, 0] <= hi)) and np.all(s[:, 1:] == 0)
        assert s[:, 0].min() < -0.59 and s[:, 0].max() > -0.41
        if env_id == "MountainCarContinuous-v0":
            assert np.array_equal(s, s.astype(np.float32).astype(np.float64))
        assert np.array_equal(obs, s[:, :2].astype(np.float32))


@pytest.mark.parametrize("env_id", IDS)
def test_device_time_limits(env_id):
    """Constant actions that never reach the goal truncate exactly at the time limit and never terminate."""
    from diamond.envs import DeviceVectorEnv
    N_ = 64
    env = DeviceVectorEnv(env_id, N_, seed=2)
    action = np.zeros((N_, 1), np.float32) if env_id == "MountainCarContinuous-v0" else np.ones(N_, np.int64)
    for t in range(LIMIT[env_id]):
        _, _, term, trunc, _ = env.step(action)
        assert not term.any()
        assert trunc.all() == (t == LIMIT[env_id] - 1) and trunc.any() == trunc.all()
    assert torch.all(env.steps == LIMIT[env_id])


def test_device_discrete_envs_refuse_bad_actions_and_descriptors():
    from diamond import _native
    from diamond.envs import DeviceVectorEnv
    for env_id in ("Acrobot-v1", "MountainCar-v0"):
        env = DeviceVectorEnv(env_id, 8, seed=0)
        before = env.state.clone()
        for bad in (-1, 3):
            a = np.ones(8, np.int64)
            a[3] = bad
            with pytest.raises(ValueError):
                env.step(a)
        assert torch.equal(env.state, before)
    env = DeviceVectorEnv("Acrobot-v1", 8, seed=0)
    for kind, D, A, what in ((4, 6, 2, "expected 3"), (4, 4, 3, "expected 6"), (5, 2, 1, "expected 3"), (6, 2, 3, "expected 1"),
                             (6, 3, 1, "expected 2")):
        desc = _native.EnvDesc(kind, 8, D, A, 0, 0, 0.0, 0.0)
        with pytest.raises(_native.NativeError, match=what):
            env.ctx.env_reset(desc, env._st, None)


def _agent(agent_name, env_id, N_, T, seed, **cfg_kw):
    import diamond
    from diamond.envs import DeviceVectorEnv
    Agent, Cfg = getattr(diamond, agent_name), getattr(diamond, agent_name + "Config")
    cfg = Cfg(num_envs=N_, rollout_steps=T, verbose=False, seed=seed, **cfg_kw)
    agent = Agent(DeviceVectorEnv.factory(env_id, seed=seed), cfg)
    agent.current_observations, _ = agent.envs.reset(seed=seed)
    if agent_name == "RecurrentPPO":
        agent.prev_dones = np.zeros(N_, dtype=bool)
        agent.current_hx = torch.zeros(1, N_, cfg.gru_hidden_dim, device=agent.device)
    return agent


@pytest.mark.parametrize("agent_name,env_id", AGENT_PAIRS)
def test_rollout_on_new_device_envs_keeps_rollout_semantics_and_learns(agent_name, env_id):
    """obs[t+1] is next_obs[t] unless the environment finished at t (then a freshly reset observation), finished steps carry the
    id's termination / time-limit flags, and learn() on the buffer changes the parameters."""
    N_, T = 64, 128
    agent = _agent(agent_name, env_id, N_, T, 3, total_steps=N_ * T * 8)
    first = agent.envs.cur_obs.clone()
    agent.envs.steps[: N_ // 2] = LIMIT[env_id] - 40                 # half the environments truncate inside this rollout
    buf = agent.rollout()
    torch.cuda.synchronize()
    assert torch.equal(buf.obs[0], first)
    done = (buf.terminations + buf.truncations) > 0
    assert done[:, : N_ // 2].any(0).all()
    cont_rows = ~done[:-1]
    assert torch.equal(buf.obs[1:][cont_rows], buf.next_obs[:-1][cont_rows])
    assert not torch.equal(buf.obs[1:][done[:-1]], buf.next_obs[:-1][done[:-1]])
    assert torch.equal(agent.envs.cur_obs[~done[-1]], buf.next_obs[-1][~done[-1]])
    assert not ((buf.terminations > 0) & (buf.truncations > 0)).any()
    if env_id == "Acrobot-v1":
        nobs = buf.next_obs.double()
        tip = -nobs[..., 0] - (nobs[..., 0] * nobs[..., 2] - nobs[..., 1] * nobs[..., 3])      # -cos th1 - cos(th1 + th2)
        term = buf.terminations > 0
        assert torch.all(tip[term] > 1.0 - 1e-5) and torch.all(tip[~term] < 1.0 + 1e-5)
        assert torch.all(buf.rewards == torch.where(term, 0.0, -1.0))
    elif env_id == "MountainCar-v0":                                   # float32 observations of the float64 state: one direction
        assert torch.all(buf.rewards == -1.0)
        goal = (buf.next_obs[..., 0] >= 0.5) & (buf.next_obs[..., 1] >= 0)
        assert torch.all(goal[buf.terminations > 0])
    else:
        assert torch.equal(buf.terminations > 0, (buf.next_obs[..., 0] >= 0.45) & (buf.next_obs[..., 1] >= 0))
    if agent_name == "RecurrentPPO":
        assert torch.equal(buf.prev_dones[1:], done[:-1])
    before = {k: v.detach().clone() for k, v in agent.network.state_dict().items()}
    agent.learn(buf)
    assert torch.isfinite(agent.last_losses).all()
    assert any(not torch.equal(before[k], v) for k, v in agent.network.state_dict().items())


@pytest.mark.parametrize("agent_name,env_id", AGENT_PAIRS)
def test_new_device_env_rollout_graph_replay_is_bit_identical_to_eager(agent_name, env_id):
    """From the third rollout the T x (forward, sampling, environment) launches replay as one CUDA graph; buffers, environment state
    and the parameters after learn() equal the eagerly launched run bit for bit."""
    N_, T = 64, 32
    recurrent = agent_name == "RecurrentPPO"
    keys = (("obs", "actions", "rewards", "terminations", "truncations", "prev_dones", "log_probs", "values", "next_values", "hx0")
            if recurrent else ("obs", "next_obs", "actions", "rewards", "terminations", "truncations", "values", "logp"))

    def run(use_graphs):
        agent = _agent(agent_name, env_id, N_, T, 13, total_steps=T * N_ * 16)
        agent.engine.use_graphs = use_graphs
        agent.envs.steps[::3] = LIMIT[env_id] - 50                   # episodes end inside the captured rollouts
        out = []
        for it in range(5):
            buf = agent.rollout()
            out.append([getattr(buf, k).clone() for k in keys] + [agent.envs.state.clone(), agent.envs.cur_obs.clone()])
            np.random.seed(it)
            agent.learn(buf)
            out[-1].append(torch.cat([q.detach().flatten() for q in agent.network.parameters()]).clone())
        replayed = (agent._ro_graph if recurrent else agent._rollout_graph) is not None
        return out, replayed

    (a, ra), (b, rb) = run(True), run(False)
    assert ra and not rb
    for it, (xa, xb) in enumerate(zip(a, b)):
        for k, (u, v) in enumerate(zip(xa, xb)):
            assert torch.equal(u, v), (it, k)


@pytest.mark.parametrize("env_id,N_,T,rollouts", [("Acrobot-v1", 64, 128, 5), ("MountainCar-v0", 64, 128, 3),
                                                  ("MountainCarContinuous-v0", 16, 256, 5)])
def test_new_device_env_episode_statistics_equal_host_ticker(env_id, N_, T, rollouts):
    """The device-side episode statistics leave the Ticker where the reference's per-step `ticker.tick(rewards, dones)` leaves it."""
    from diamond.utils import Ticker
    agent = _agent("ContinuousPPO" if env_id == "MountainCarContinuous-v0" else "PPO", env_id, N_, T, 3, total_steps=T * N_ * 100)
    host = Ticker(agent.cfg.total_steps, N_, T, verbose=False)
    for _ in range(rollouts):
        buf = agent.rollout()
        rew = buf.rewards.double().cpu().numpy()
        dones = ((buf.terminations + buf.truncations) > 0).cpu().numpy()
        for t in range(T):
            host.tick(rew[t], dones[t])
    got, ref = agent.ticker.logs, host.logs
    assert ref["total_episodes"] > 0
    assert got["total_steps"] == ref["total_steps"] and got["total_episodes"] == ref["total_episodes"]
    assert got["episode_lengths"] == ref["episode_lengths"]
    assert got["episode_returns"] == ref["episode_returns"]
    np.testing.assert_array_equal(agent._epstats["ep_len"].cpu().numpy(), host.current_lengths)
    np.testing.assert_array_equal(agent._epstats["ep_return"].cpu().numpy(), host.current_returns)


def test_ppo_learns_acrobot_on_device():
    """End-to-end train() on device-resident Acrobot-v1 with the default hyper-parameters: the mean length of the last 100 episodes
    falls well below the 500-step cap that a random policy mostly hits.  Budget and bound: ACROBOT_ROLLOUTS / ACROBOT_MAX_MEAN_LENGTH,
    with the measured curves they were chosen from, at the top of this file."""
    from diamond import PPO, PPOConfig
    from diamond.envs import DeviceVectorEnv
    cfg = PPOConfig(num_envs=64, rollout_steps=128, verbose=False, seed=1, total_steps=64 * 128 * ACROBOT_ROLLOUTS)
    agent = PPO(DeviceVectorEnv.factory("Acrobot-v1", seed=1), cfg)
    agent.train()
    lengths = list(agent.ticker.recent_lengths)
    assert len(lengths) == 100 and np.mean(lengths) < ACROBOT_MAX_MEAN_LENGTH, np.mean(lengths)


@pytest.mark.parametrize("agent_name,env_id", [("PPO", "Acrobot-v1"), ("ContinuousPPO", "MountainCarContinuous-v0")])
def test_host_path_runs_new_ids(agent_name, env_id):
    """The same ids through diamond.envs.make and the host SyncVectorEnv: one rollout and one learn()."""
    import diamond
    from diamond import envs
    Agent, Cfg = getattr(diamond, agent_name), getattr(diamond, agent_name + "Config")
    cfg = Cfg(num_envs=4, rollout_steps=32, verbose=False, seed=2, total_steps=4 * 32 * 4)
    agent = Agent(lambda: envs.make(env_id), cfg)
    agent.current_observations, _ = agent.envs.reset(seed=2)
    buf = agent.rollout()
    before = torch.cat([q.detach().flatten() for q in agent.network.parameters()]).clone()
    agent.learn(buf)
    torch.cuda.synchronize()
    assert torch.isfinite(agent.last_losses).all()
    assert not torch.equal(before, torch.cat([q.detach().flatten() for q in agent.network.parameters()]))
