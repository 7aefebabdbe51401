"""GPU: per-environment observation and reward normalisation inside the device environments (csrc/envs.cu, DeviceVectorEnv's
normalize_observation / normalize_reward) against the float64 restatement of Gymnasium's wrappers (tests/normalize_oracle.py).

The oracle is fed with the raw stream of an identical environment without normalisation (the dynamics do not depend on it).  Rewards
enter the oracle in float64 as the kernel computes them: for the classic kinds the reference environment runs host-array steps
with its running return zeroed before each step, so afterwards `ep_return` holds exactly the step's float64 reward."""
import os
import sys
import types

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import normalize_oracle as NO  # noqa: E402

pytestmark = pytest.mark.gpu

LIMIT = {"CartPole-v1": 500, "Pendulum-v1": 200, "Acrobot-v1": 500, "MountainCar-v0": 200, "MountainCarContinuous-v0": 999}
KINDS = [("CartPole-v1", {}), ("Pendulum-v1", {}), ("Acrobot-v1", {}), ("MountainCar-v0", {}), ("MountainCarContinuous-v0", {}),
         ("Synthetic", dict(obs_dim=67, n_actions=3, p_term=0.02, p_trunc=0.01)),
         ("Synthetic", dict(obs_dim=5, n_actions=2, continuous=True, p_term=0.02, p_trunc=0.01))]
STATS = ("obs_mean", "obs_var", "obs_count", "return_stats")


def _assert_f32(got, exp, what):
    """float32 arrays equal up to one ulp (the allowance of the MountainCarContinuous check for CUDA's and libm's cos)."""
    got, exp = np.asarray(got, np.float32), np.asarray(exp, np.float32)
    assert got.shape == exp.shape, what
    ulps = np.abs(got.view(np.int32).astype(np.int64) - exp.view(np.int32).astype(np.int64))
    assert ulps.max(initial=0) <= 1, (what, int(ulps.max()), np.argwhere(ulps > 1)[:4])


def _assert_stats(env, oracle, what):
    for k in STATS:
        np.testing.assert_array_equal(getattr(env, k).cpu().numpy(), getattr(oracle, k), err_msg=f"{what}: {k}")


def _actions(env, rng):
    if env.continuous:
        return rng.uniform(-2.5, 2.5, (env.num_envs, env.act_dim)).astype(np.float32)
    return rng.integers(0, env.act_dim, env.num_envs)


def _buffer(env, T):
    f = dict(dtype=torch.float32, device=env.device)
    N_, D = env.num_envs, env.obs_dim
    return types.SimpleNamespace(obs=torch.empty(T, N_, D, **f), next_obs=torch.empty(T, N_, D, **f),
                                 actions=torch.empty(T, N_, env.act_dim, **f) if env.continuous else torch.empty(T, N_, dtype=torch.int32, device=env.device),
                                 rewards=torch.empty(T, N_, **f), terminations=torch.empty(T, N_, **f), truncations=torch.empty(T, N_, **f),
                                 raw_rewards=torch.empty(T, N_, **f), filled=0)


@pytest.mark.parametrize("path", ["step_into", "host"])
@pytest.mark.parametrize("env_id,kw", KINDS, ids=[k[0] + ("-cont" if k[1].get("continuous") else "") for k in KINDS])
def test_device_normalisation_matches_per_env_wrappers(env_id, kw, path):
    """600 random steps with resets, through step_into (in-kernel resets) or host step / reset(mask), with the statistics frozen for
    100 of them: statistics and accumulators bit-identical to the oracle, normalised observations (final and post-reset) and rewards
    equal to its float32 casts, raw rewards equal to the unnormalised environment's, next_obs[t] == obs[t + 1] where not done."""
    from diamond.envs import DeviceVectorEnv
    N_, T, gamma = 64, 600, 0.95
    clip_o, clip_r = (4.0, 3.0) if path == "host" else (None, None)
    classic = env_id in LIMIT
    raw = DeviceVectorEnv(env_id, N_, seed=7, **kw)
    nrm = DeviceVectorEnv(env_id, N_, seed=7, normalize_observation=True, normalize_reward=True, gamma=gamma, clip_observation=clip_o,
                          clip_reward=clip_r, **kw)
    assert torch.all(nrm.obs_count == 1e-4) and torch.all(nrm.obs_mean == 0)      # the constructor's reset counts nothing
    assert nrm.single_observation_space.shape == (raw.obs_dim,) and np.all(np.isinf(nrm.single_observation_space.high))
    oracle = NO.PerEnvNormalizer(N_, raw.obs_dim, gamma=gamma, clip_observation=clip_o, clip_reward=clip_r)
    o_raw, _ = raw.reset(seed=11)
    o_n, _ = nrm.reset(seed=11)
    _assert_f32(o_n, oracle.observe(o_raw), "reset(seed)")
    if classic:
        for env in (raw, nrm):
            env.steps[::4] = LIMIT[env_id] - 30 - torch.arange(0, N_, 4, device=env.device, dtype=torch.int32) % 7
    rbuf = _buffer(raw, T) if (path == "step_into" and not classic) else None
    buf = _buffer(nrm, T) if path == "step_into" else None
    rng = np.random.default_rng(3)
    resets = 0
    for t in range(T):
        if t in (300, 400):
            nrm.update_running_mean = oracle.update_running_mean = t == 400
        if env_id == "MountainCarContinuous-v0" and t % 100 == 50:  # send every eighth car to the goal
            for env in (raw, nrm):
                env.state[::8, 0], env.state[::8, 1] = float(np.float32(0.449)), float(np.float32(0.05))
        a = _actions(raw, rng)
        if rbuf is None:                                               # reference: host-array steps
            if classic:
                raw.ep_return.zero_()
            o1, r1, te1, tr1, _ = raw.step(a)
            r64 = raw.ep_return.cpu().numpy() if classic else r1
            dones = te1 | tr1
            post = raw.reset(options={"reset_mask": dones})[0] if dones.any() else None
        else:                                                          # synthetic in-kernel resets draw differently: same path
            raw.step_into(rbuf, t, a)
            o1, r64 = rbuf.next_obs[t].cpu().numpy(), rbuf.rewards[t].double().cpu().numpy()
            te1, tr1 = rbuf.terminations[t].cpu().numpy() > 0, rbuf.truncations[t].cpu().numpy() > 0
            dones = te1 | tr1
            post = raw.cur_obs.cpu().numpy()
        exp_final = oracle.observe(o1)
        exp_rew = oracle.reward(r64, te1).astype(np.float32)
        if path == "host":
            o2, r2, te2, tr2, info = nrm.step(a)
            np.testing.assert_array_equal(te2, te1)
            np.testing.assert_array_equal(tr2, tr1)
            _assert_f32(o2, exp_final, f"final obs, step {t}")
            _assert_f32(r2.astype(np.float32), exp_rew, f"reward, step {t}")
            np.testing.assert_array_equal(info["raw_rewards"], r64.astype(np.float32).astype(np.float64))
            if dones.any():
                p2, _ = nrm.reset(options={"reset_mask": dones})
                _assert_f32(p2[dones], oracle.observe(post, dones)[dones], f"reset obs, step {t}")
                _assert_f32(p2[~dones], exp_final[~dones], f"untouched obs, step {t}")
        else:
            nrm.step_into(buf, t, a)
            np.testing.assert_array_equal(buf.terminations[t].cpu().numpy() > 0, te1)
            _assert_f32(buf.next_obs[t].cpu().numpy(), exp_final, f"final obs, step {t}")
            _assert_f32(buf.rewards[t].cpu().numpy(), exp_rew, f"reward, step {t}")
            np.testing.assert_array_equal(buf.raw_rewards[t].cpu().numpy(), r64.astype(np.float32))
            exp_cur = exp_final.copy()
            if dones.any():
                exp_cur[dones] = oracle.observe(post, dones)[dones]
            _assert_f32(nrm.cur_obs.cpu().numpy(), exp_cur, f"cur_obs, step {t}")
            assert torch.equal(nrm.cur_obs[torch.as_tensor(~dones, device=nrm.device)], buf.next_obs[t][torch.as_tensor(~dones, device=nrm.device)])
        resets += int(dones.sum())
        if t % 50 == 49 or t == T - 1:
            _assert_stats(nrm, oracle, f"step {t}")
    assert resets > 0
    if buf is not None:                                                # next_obs[t] is obs[t + 1] wherever the env did not finish
        done = ((buf.terminations + buf.truncations) > 0)[:-1]
        assert torch.equal(buf.obs[1:][~done], buf.next_obs[:-1][~done])


def test_normalisation_refuses_bad_descriptors_before_launching():
    from diamond import _native as N
    from diamond.envs import DeviceVectorEnv
    env = DeviceVectorEnv("CartPole-v1", 8, seed=0, normalize_observation=True, normalize_reward=True)
    before = {k: getattr(env, k).clone() for k in env.state_tensors}
    good = env.desc
    for field, value, msg in (("gamma", 1.5, "gamma"), ("gamma", -0.1, "gamma"), ("epsilon", 0.0, "epsilon"), ("clip_reward", -1.0, "clip"),
                              ("clip_observation", -1.0, "clip"), ("normalize", 4, "flags")):
        d = N.EnvDesc.from_buffer_copy(good)
        setattr(d, field, value)
        with pytest.raises(N.NativeError, match=msg):
            env.ctx.env_reset(d, env._st, None)
    for field, msg in (("obs_mean", "obs_mean"), ("ret_stats", "ret_stats"), ("update", "update flag")):
        st = N.EnvState.from_buffer_copy(env._st)
        setattr(st, field, None)
        with pytest.raises(N.NativeError, match=msg):
            env.ctx.env_reset(good, st, None)
    torch.cuda.synchronize()
    for k, v in before.items():
        assert torch.equal(getattr(env, k), v), k
    with pytest.raises(ValueError):
        DeviceVectorEnv("CartPole-v1", 8, normalize_reward=True, gamma=2.0)
    with pytest.raises(ValueError):
        DeviceVectorEnv("CartPole-v1", 8, normalize_observation=True, clip_observation=0.0)


@pytest.mark.parametrize("env_id,kw", [("CartPole-v1", {}), ("Synthetic", dict(obs_dim=64, n_actions=4, continuous=True))])
def test_env_sharding_needs_no_exchange(env_id, kw):
    """Statistics belong to global environment ids: one environment of 2n equals two of n with env_offset 0 and n, bit for bit."""
    from diamond.envs import DeviceVectorEnv
    n, T = 32, 300
    norm = dict(normalize_observation=True, normalize_reward=True, gamma=0.9)
    full = DeviceVectorEnv(env_id, 2 * n, seed=4, **norm, **kw)
    halves = [DeviceVectorEnv(env_id, n, seed=4, env_offset=k * n, **norm, **kw) for k in (0, 1)]
    envs = [full] + halves
    for e in envs:
        e.reset(seed=4)
        if env_id in LIMIT:
            e.steps.fill_(LIMIT[env_id] - 100)
    bufs = [_buffer(e, T) for e in envs]
    rng = np.random.default_rng(0)
    for t in range(T):
        a = _actions(full, rng)
        full.step_into(bufs[0], t, a)
        halves[0].step_into(bufs[1], t, a[:n])
        halves[1].step_into(bufs[2], t, a[n:])
    torch.cuda.synchronize()
    assert (bufs[0].terminations + bufs[0].truncations).sum() > 0
    for k in ("obs", "next_obs", "rewards", "raw_rewards", "terminations", "truncations"):
        assert torch.equal(getattr(bufs[0], k), torch.cat([getattr(bufs[1], k), getattr(bufs[2], k)], 1)), k
    for k in full.state_tensors:
        assert torch.equal(getattr(full, k), torch.cat([getattr(halves[0], k), getattr(halves[1], k)], 0)), k


def _agent(agent_name, env_id, N_, T, seed, env_kw, network_cls=None, **cfg_kw):
    import diamond
    from diamond.envs import DeviceVectorEnv
    Agent, Cfg = getattr(diamond, agent_name), getattr(diamond, agent_name + "Config")
    cfg = Cfg(num_envs=N_, rollout_steps=T, verbose=False, seed=seed, **cfg_kw)
    args = {} if network_cls is None else dict(network_cls=network_cls)
    agent = Agent(DeviceVectorEnv.factory(env_id, seed=seed, **env_kw), cfg, **args)
    agent.current_observations, _ = agent.envs.reset(seed=seed)
    if agent_name.startswith("Recurrent"):
        agent.prev_dones = np.zeros(N_, dtype=bool)
        agent.current_hx = torch.zeros(1, N_, cfg.gru_hidden_dim, device=agent.device)
    return agent


@pytest.mark.parametrize("agent_name,env_id", [("PPO", "CartPole-v1"), ("RecurrentContinuousPPO", "Pendulum-v1")])
def test_graph_replayed_rollouts_equal_eager_and_follow_the_freeze_flag(agent_name, env_id):
    """Rollouts replayed as one CUDA graph equal eagerly launched ones bit for bit (buffers, raw rewards, environment state, statistics,
    parameters after learn()); update_running_mean = False set between replays freezes the statistics of the next replays, True
    resumes them."""
    N_, T = 64, 32
    recurrent = agent_name.startswith("Recurrent")
    keys = (("obs", "actions", "rewards", "raw_rewards", "terminations", "truncations", "log_probs", "values", "next_values")
            if recurrent else ("obs", "next_obs", "actions", "rewards", "raw_rewards", "terminations", "truncations", "values", "logp"))
    norm = dict(normalize_observation=True, normalize_reward=True, clip_observation=10.0, clip_reward=10.0)

    def run(use_graphs):
        agent = _agent(agent_name, env_id, N_, T, 13, norm, total_steps=T * N_ * 16)
        agent.engine.use_graphs = use_graphs
        agent.envs.steps[::3] = LIMIT[env_id] - 50
        out = []
        for it in range(6):
            if it in (3, 5):
                agent.envs.update_running_mean = it == 5
            buf = agent.rollout()
            envs = agent.envs
            out.append([getattr(buf, k).clone() for k in keys] + [getattr(envs, k).clone() for k in envs.state_tensors])
            np.random.seed(it)
            agent.learn(buf)
            out[-1].append(torch.cat([q.detach().flatten() for q in agent.network.parameters()]).clone())
        replayed = (agent._ro_graph if recurrent else agent._rollout_graph) is not None
        return out, replayed, agent.envs.state_tensors

    (a, ra, names), (b, rb, _) = run(True), run(False)
    assert ra and not rb
    for it, (xa, xb) in enumerate(zip(a, b)):
        for k, (u, v) in enumerate(zip(xa, xb)):
            assert torch.equal(u, v), (it, k)
    s = {name: [a[it][len(keys) + j] for it in range(6)] for j, name in enumerate(names)}
    for name in ("obs_mean", "obs_var", "obs_count"):
        assert not torch.equal(s[name][1], s[name][2]), name             # replays update ...
        assert torch.equal(s[name][2], s[name][3]) and torch.equal(s[name][3], s[name][4]), name     # ... frozen ones do not
        assert not torch.equal(s[name][4], s[name][5]), name
    rs = s["return_stats"]
    assert torch.equal(rs[2][:, 1:], rs[4][:, 1:]) and not torch.equal(rs[4][:, 1:], rs[5][:, 1:])
    assert not torch.equal(rs[3][:, 0], rs[4][:, 0])                  # the accumulator runs while frozen


def _custom_mlp():
    from diamond.networks import ActorCriticNetwork

    class Custom(ActorCriticNetwork):                                  # not the default network: the host rollout loop
        pass
    return Custom


@pytest.mark.parametrize("agent_name,env_id,custom", [("PPO", "CartPole-v1", False), ("PPO", "CartPole-v1", True),
                                                      ("RecurrentContinuousPPO", "Pendulum-v1", False)])
def test_ticker_reports_raw_returns(agent_name, env_id, custom):
    """With reward normalisation the Ticker reports the raw episode returns: equal to those of an otherwise identical run without it
    (rollouts only, so both runs take the same actions)."""
    N_, T, R = 32, 64, 8
    logs = []
    for norm in (False, True):
        agent = _agent(agent_name, env_id, N_, T, 21, dict(normalize_reward=norm, gamma=0.9),
                       network_cls=_custom_mlp() if custom else None, total_steps=N_ * T * 100)
        if env_id == "CartPole-v1":
            agent.envs.steps[::2] = 480
        for _ in range(R):
            buf = agent.rollout()
        if norm and not custom:
            assert not torch.equal(buf.rewards, buf.raw_rewards)
        logs.append(agent.ticker.logs)
    assert logs[0]["total_episodes"] > 0
    for k in ("total_steps", "total_episodes", "episode_returns", "episode_lengths"):
        assert logs[0][k] == logs[1][k], k


def test_train_resume_with_normalisation_is_bit_identical(tmp_path):
    """train(resume_from=...) restores the statistics and the freeze flag: interrupted + resumed equals uninterrupted, bit for bit."""
    from diamond import ContinuousPPO, ContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.utils import Checkpointer
    N_, T, R = 64, 32, 7

    def make(tag):
        cfg = ContinuousPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=5, total_steps=N_ * T * R, num_minibatches=4)
        agent = ContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=5, normalize_observation=True, normalize_reward=True,
                                                      clip_observation=10.0, clip_reward=10.0), cfg)
        agent.checkpointer = Checkpointer(tmp_path / tag, "run")
        return agent

    full = make("full")
    full.train()
    part = make("part")
    part.train(max_rollouts=3)
    resumed = make("resumed")
    resumed.train(resume_from=part.last_checkpoint)
    torch.cuda.synchronize()
    assert torch.equal(resumed.engine.P, full.engine.P)
    for k in full.envs.state_tensors:
        assert torch.equal(getattr(resumed.envs, k), getattr(full.envs, k)), k
    assert not torch.equal(part.envs.obs_mean, full.envs.obs_mean)
    a, b = resumed.ticker.logs, full.ticker.logs
    for k in ("total_steps", "total_episodes", "episode_returns", "episode_lengths"):
        assert a[k] == b[k], k
    # the freeze flag travels with the checkpoint
    part.envs.update_running_mean = False
    st = part._train_state(3)
    fresh = make("fresh")
    fresh._restore_train_state(st)
    assert fresh.envs.update_running_mean is False and int(fresh.envs._update.item()) == 0
    for k in part.envs.state_tensors:
        assert torch.equal(getattr(fresh.envs, k), getattr(part.envs, k)), k


# Learning on device Pendulum-v1 (tests/env_normalize_learning_curve.py, one B200 at a 1000 W power limit, 5 seeds, observations and
# rewards normalised and clipped to +-10): RecurrentContinuousPPO at its defaults (32 x 32, gamma 0.99, lr 3e-4) goes from about
# -1200 to -227 ... -314 (mean of the last 20 rollouts at 600 rollouts); every seed is above -600 from rollout 480 on (about 1.7 s for
# 600 rollouts).  The same runs without normalisation stay between -1154 and -1355 in every window.  Budget 600 rollouts, bound -600.
LEARN_ROLLOUTS, LEARN_BOUND = 600, -600.0


def test_agent_learns_device_pendulum_with_normalisation():
    """The measured setting where normalisation makes the agent learn: the mean raw return of the Ticker's last 100 episodes passes a
    bound that runs without normalisation and random policies do not reach."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    cfg = RecurrentContinuousPPOConfig(verbose=False, seed=0)
    cfg.total_steps = cfg.num_envs * cfg.rollout_steps * LEARN_ROLLOUTS
    agent = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=0, normalize_observation=True, normalize_reward=True,
                                                           gamma=cfg.gamma, clip_observation=10.0, clip_reward=10.0), cfg)
    agent.train()
    returns = list(agent.ticker.recent_returns)
    assert len(returns) > 0 and np.mean(returns) > LEARN_BOUND, np.mean(returns)
