"""GPU: predict() / evaluate() of the four agents -- the greedy kernel, the evaluation bookkeeping kernel, the device evaluation
loop against a host loop over predict(), graph replay, and that evaluating leaves training bit-identical."""
import numpy as np
import pytest
import torch

from evaluate_oracle import EvalBook, quotas

pytestmark = pytest.mark.gpu


def _ctx():
    from diamond import _native
    return _native.get_context()


# ---- greedy kernel -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("A", [1, 2, 3, 31, 32, 33, 100, 1024])
@pytest.mark.parametrize("N", [1, 129, 1000])
def test_greedy_kernel_is_torch_argmax_on_adversarial_logits(N, A):
    """Ties at every position (logits drawn from four values), +-inf, rows of -inf only, NaN rows (one NaN, several, all NaN)."""
    ctx = _ctx()
    rng = np.random.default_rng(N * 1031 + A)
    z = rng.choice(np.array([-1.0, 0.0, 2.5, 2.5], np.float32), size=(N, A))
    kind = rng.integers(0, 6, N)
    for e in range(N):
        k = kind[e]
        if k == 1:
            z[e, rng.integers(0, A, rng.integers(1, 3))] = np.inf
        elif k == 2:
            z[e, rng.integers(0, A, rng.integers(1, 3))] = -np.inf
        elif k == 3:
            z[e] = -np.inf
        elif k == 4:
            z[e, rng.integers(0, A, rng.integers(1, 4))] = np.nan
        elif k == 5 and e % 2:
            z[e] = np.nan
    logits = torch.as_tensor(z).cuda()
    got = ctx.select_greedy_categorical(logits)
    torch.cuda.synchronize()
    ref = torch.argmax(torch.as_tensor(z), -1)
    assert got.dtype == torch.int64 and torch.equal(got.cpu(), ref)
    assert torch.equal(got, torch.argmax(logits, -1))


@pytest.mark.parametrize("A", [2, 7, 100])
def test_greedy_log_prob_is_the_sampling_kernels_formula(A):
    """Wherever the sampling kernel drew the greedy action, both kernels' log-probs are bit-identical (same formula); all of them
    agree with float64 log_softmax."""
    ctx = _ctx()
    rng = np.random.default_rng(A)
    N = 4099
    logits = torch.as_tensor(rng.standard_normal((N, A)).astype(np.float32) * 3).cuda()
    lp_g, lp_s = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
    greedy = ctx.select_greedy_categorical(logits, log_probs=lp_g)
    sampled = ctx.sample_categorical(logits, 7, 0, 0, log_probs=lp_s)
    torch.cuda.synchronize()
    same = greedy == sampled
    assert int(same.sum()) > N // (2 * A)
    assert torch.equal(lp_g[same], lp_s[same])
    ref = torch.log_softmax(logits.double(), -1).gather(1, greedy[:, None])[:, 0]
    assert float((lp_g.double() - ref).abs().max()) < 1e-5


# ---- bookkeeping kernel ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,T,chunks,kmax", [(1, 16, 3, 2), (300, 32, 5, 4), (1000, 7, 9, 3)])
def test_eval_episodes_kernel_matches_numpy_restatement(N, T, chunks, kmax):
    ctx = _ctx()
    rng = np.random.default_rng(N + T)
    q = rng.integers(0, kmax + 1, N).astype(np.int32)               # quotas 0 .. kmax
    book = EvalBook(q)
    dev = lambda x: torch.as_tensor(x).cuda()
    slot = dev(book.slot)
    ep_return, ep_len = torch.zeros(N, dtype=torch.float64, device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda")
    rec = torch.zeros(N, dtype=torch.int32, device="cuda")
    E = max(int(q.sum()), 1)
    out_r, out_l = torch.full((E,), -1.0, dtype=torch.float64, device="cuda"), torch.full((E,), -1, dtype=torch.int32, device="cuda")
    remaining = torch.tensor([book.remaining], dtype=torch.int32, device="cuda")
    for c in range(chunks):
        r = (rng.standard_normal((T, N)) * 10).astype(np.float32)
        p = 0.02 + 0.2 * rng.random(N)                                # episodes of very different lengths, many straddle chunks
        term = (rng.random((T, N)) < p).astype(np.float32)
        trunc = ((rng.random((T, N)) < 0.03) & (term == 0)).astype(np.float32)
        ctx.eval_episodes(dev(r), dev(term), dev(trunc), dev(q), slot, ep_return, ep_len, rec, out_r, out_l, remaining)
        book.chunk(r, term, trunc)
        torch.cuda.synchronize()
        assert np.array_equal(rec.cpu().numpy(), book.recorded)
        assert int(remaining.item()) == book.remaining
        assert np.array_equal(ep_return.cpu().numpy(), book.ep_return) and np.array_equal(ep_len.cpu().numpy(), book.ep_len)
    n_out = int(q.sum())
    filled = np.zeros(n_out, dtype=bool)                              # slots of episodes recorded; the others are never written
    for e in range(N):
        filled[book.slot[e]:book.slot[e] + book.recorded[e]] = True
    got_r, got_l = out_r.cpu().numpy()[:n_out], out_l.cpu().numpy()[:n_out].astype(np.int64)
    assert np.array_equal(got_r[filled], book.out_returns[filled]) and np.array_equal(got_l[filled], book.out_lengths[filled])
    assert (got_r[~filled] == -1.0).all() and (got_l[~filled] == -1).all()
    assert book.remaining < int((q > 0).sum())                         # some environments did reach their quota


# ---- predict() on the default networks against float64 ---------------------------------------------------------------------
def _near_tie(l64, tol):
    top2 = torch.topk(l64, 2, dim=-1).values
    return (top2[:, 0] - top2[:, 1]) <= tol


@pytest.mark.parametrize("H,A", [(64, 2), (1024, 4), (256, 100), (64, 33)])
def test_predict_is_argmax_of_float64_logits_mlp(H, A):
    """Fused forward (SIMT, tensor-core trunk, GEMM heads) + greedy kernel against argmax of the float64 torch module.  Rows whose
    top two float64 logits lie within twice the forward's tolerance (1e-5 of max |logit|) are exempt."""
    from diamond import PPO, PPOConfig, envs
    from diamond.networks import ActorCriticNetwork
    D, n = 24, 2048
    cfg = PPOConfig(num_envs=2, rollout_steps=8, network_hidden_dim=H, verbose=False, seed=2)
    agent = PPO(lambda: envs.SyntheticEnv(D, A), cfg)
    with torch.no_grad():
        agent.network.actor_head[2].weight.mul_(300.0)               # spread the logits: the default gain 0.01 makes most rows ties
    rng = np.random.default_rng(H + A)
    obs = rng.standard_normal((n, D)).astype(np.float32)
    got_host = agent.predict(obs)
    got_dev = agent.predict(torch.as_tensor(obs).cuda())
    assert isinstance(got_host, np.ndarray) and got_host.dtype == np.int64 and torch.is_tensor(got_dev) and got_dev.is_cuda
    assert np.array_equal(got_host, got_dev.cpu().numpy())
    ref = ActorCriticNetwork(agent.envs.single_observation_space, agent.envs.single_action_space, cfg).double()
    ref.load_state_dict({k: v.detach().cpu().double() for k, v in agent.network.state_dict().items()})
    with torch.no_grad():
        l64, _ = ref.get_logits_and_values(torch.as_tensor(obs).double())
    exempt = _near_tie(l64, 2e-5 * float(l64.abs().max()))
    assert int(exempt.sum()) < n // 20
    assert torch.equal(torch.as_tensor(got_host)[~exempt], torch.argmax(l64, -1)[~exempt])


def test_predict_is_argmax_of_float64_logits_gru():
    """RecurrentPPO's fused GRU step + greedy kernel over 8 steps with random resets, against the float64 module carrying its own
    float64 hidden state."""
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    from diamond.recurrent import RecurrentActorCriticNetwork
    D, A, n = 6, 5, 1024
    cfg = RecurrentPPOConfig(num_envs=2, rollout_steps=8, verbose=False, seed=3)
    agent = RecurrentPPO(lambda: envs.SyntheticEnv(D, A), cfg)
    with torch.no_grad():
        agent.network.actor_head[2].weight.mul_(300.0)
    ref = RecurrentActorCriticNetwork(agent.envs.single_observation_space, agent.envs.single_action_space, cfg).double()
    ref.load_state_dict({k: v.detach().cpu().double() for k, v in agent.network.state_dict().items()})
    rng = np.random.default_rng(0)
    hx, h64 = None, torch.zeros(1, n, cfg.gru_hidden_dim, dtype=torch.float64)
    exempt_total = 0
    for t in range(8):
        obs = rng.standard_normal((n, D)).astype(np.float32)
        dones = rng.random(n) < 0.2
        actions, hx = agent.predict(obs, hx, dones)
        assert hx.shape == (1, n, cfg.gru_hidden_dim)
        with torch.no_grad():
            l64, _, h64 = ref.get_logits_values_and_hx(torch.as_tensor(obs).double()[None], h64, torch.as_tensor(dones)[None])
        l64 = l64[0]
        exempt = _near_tie(l64, 2e-5 * float(l64.abs().max()))
        exempt_total += int(exempt.sum())
        assert torch.equal(torch.as_tensor(actions)[~exempt], torch.argmax(l64, -1)[~exempt]), t
    assert exempt_total < 8 * n // 20


# ---- evaluate() on device environments against a host loop over predict() --------------------------------------------------
def _host_loop(agent, env_fn, num_envs, num_episodes, seed, deterministic=True):
    """Drives a new environment from env_fn through reset / step with masked resets, actions from agent.predict."""
    envs = env_fn(num_envs)
    if envs.desc.normalize:
        envs.load_frozen_statistics(agent.envs)
    book = EvalBook(quotas(num_episodes, num_envs))
    recurrent = hasattr(agent, "prev_dones") or agent.__class__.__name__.startswith("Recurrent")
    obs, _ = envs.reset(seed=seed)
    hx, prev = None, np.zeros(num_envs, dtype=bool)
    while book.remaining > 0:
        if recurrent:
            actions, hx = agent.predict(obs, hx, prev, deterministic=deterministic)
        else:
            actions = agent.predict(obs, deterministic=deterministic)
        nobs, rew, term, trunc, info = envs.step(actions)
        book.step(info.get("raw_rewards", rew), term, trunc)
        dones = term | trunc
        obs = envs.reset(options={"reset_mask": dones})[0] if dones.any() else nobs
        prev = dones
    return book.out_returns, book.out_lengths


def _agent(kind, env_id, seed=3, num_envs=16, **env_kw):
    from diamond import (PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig, RecurrentPPO, RecurrentPPOConfig, RecurrentContinuousPPO,
                         RecurrentContinuousPPOConfig)
    from diamond.envs import DeviceVectorEnv
    Agent, Cfg = {"mlp": (PPO, PPOConfig), "mlp_cont": (ContinuousPPO, ContinuousPPOConfig), "gru": (RecurrentPPO, RecurrentPPOConfig),
                  "gru_cont": (RecurrentContinuousPPO, RecurrentContinuousPPOConfig)}[kind]
    cfg = Cfg(num_envs=num_envs, rollout_steps=32, verbose=False, seed=seed, total_steps=num_envs * 32 * 100)
    env_fn = DeviceVectorEnv.factory(env_id, seed=seed, **env_kw)
    agent = Agent(env_fn, cfg)
    return agent, env_fn


def _train(agent, rollouts):
    if hasattr(agent, "prev_dones") or agent.__class__.__name__.startswith("Recurrent"):
        n = agent.cfg.num_envs
        agent.current_observations, _ = agent.envs.reset(seed=agent.cfg.seed)
        agent.prev_dones = np.zeros(n, dtype=bool)
        agent.current_hx = torch.zeros(1, n, agent.cfg.gru_hidden_dim, device=agent.device)
    else:
        agent.current_observations, _ = agent.envs.reset(seed=agent.cfg.seed)
    for _ in range(rollouts):
        agent.learn(agent.rollout())


PAIRS = [("mlp", "CartPole-v1"), ("mlp", "Acrobot-v1"), ("mlp", "MountainCar-v0"), ("mlp_cont", "Pendulum-v1"),
         ("mlp_cont", "MountainCarContinuous-v0"), ("gru", "CartPole-v1"), ("gru_cont", "Pendulum-v1")]


@pytest.mark.parametrize("kind,env_id", PAIRS)
def test_evaluate_on_device_equals_host_loop_over_predict(kind, env_id):
    agent, env_fn = _agent(kind, env_id)
    _train(agent, 2)
    res = agent.evaluate(10, num_envs=4, seed=77)
    ret, length = _host_loop(agent, env_fn, 4, 10, 77)
    assert res["returns"].dtype == np.float64 and res["lengths"].dtype == np.int64 and res["returns"].shape == (10,)
    assert np.array_equal(res["returns"], ret) and np.array_equal(res["lengths"], length)
    assert res["mean_return"] == float(ret.mean()) and res["mean_length"] == float(length.mean())


@pytest.mark.parametrize("kind,env_id", [("mlp", "CartPole-v1"), ("mlp_cont", "Pendulum-v1"), ("gru_cont", "Pendulum-v1")])
def test_evaluate_with_normalisation_equals_host_loop_and_reads_training_statistics_only(kind, env_id):
    agent, env_fn = _agent(kind, env_id, num_envs=8, normalize_observation=True, normalize_reward=True)
    _train(agent, 2)
    before = {k: getattr(agent.envs, k).clone() for k in agent.envs.state_tensors}
    res = agent.evaluate(12, num_envs=12, seed=5)                    # 12 evaluation environments take training envs i mod 8
    ret, length = _host_loop(agent, env_fn, 12, 12, 5)
    assert np.array_equal(res["returns"], ret) and np.array_equal(res["lengths"], length)
    for k, v in before.items():
        assert torch.equal(getattr(agent.envs, k), v), k
    assert agent.envs.update_running_mean


def test_evaluate_quota_split_and_more_environments_than_episodes():
    agent, env_fn = _agent("mlp", "CartPole-v1")
    for num_episodes, num_envs in ((10, 4), (7, 3), (3, 8)):
        res = agent.evaluate(num_episodes, num_envs=num_envs, seed=9)
        ret, length = _host_loop(agent, env_fn, num_envs, num_episodes, 9)
        assert res["lengths"].shape == (num_episodes,)
        assert np.array_equal(res["returns"], ret) and np.array_equal(res["lengths"], length)


def test_evaluate_stochastic_is_reproducible_and_equals_host_loop():
    agent, env_fn = _agent("mlp", "CartPole-v1")
    _train(agent, 2)
    a = agent.evaluate(12, num_envs=4, seed=21, deterministic=False)
    b = agent.evaluate(12, num_envs=4, seed=21, deterministic=False)
    c = agent.evaluate(12, num_envs=4, seed=22, deterministic=False)
    assert np.array_equal(a["returns"], b["returns"]) and np.array_equal(a["lengths"], b["lengths"])
    assert not np.array_equal(a["lengths"], c["lengths"])
    agent.evaluate(1, num_envs=1, seed=21)                           # re-keys the evaluation generator for the host loop below
    ret, length = _host_loop(agent, env_fn, 4, 12, 21, deterministic=False)
    assert np.array_equal(a["returns"], ret) and np.array_equal(a["lengths"], length)


def test_evaluate_max_steps_names_the_unfinished_environments():
    from diamond import PPO, PPOConfig, envs
    agent, _ = _agent("mlp", "MountainCar-v0", num_envs=4)           # 200-step limit; no policy reaches the goal in 50 steps
    with pytest.raises(RuntimeError, match=r"environments \[0, 1, 2, 3\] did not finish"):
        agent.evaluate(4, num_envs=4, seed=1, max_steps=50)
    res = agent.evaluate(4, num_envs=4, seed=1, max_steps=200)        # exactly enough steps: the bound is inclusive
    assert (res["lengths"] <= 200).all()
    host = PPO(lambda: envs.MountainCarEnv(), PPOConfig(num_envs=2, rollout_steps=8, verbose=False, seed=1))
    with pytest.raises(RuntimeError, match=r"environments \[0, 1\] did not finish"):
        host.evaluate(2, num_envs=2, seed=1, max_steps=50)


def test_graph_replay_equals_eager_evaluation():
    for kind, env_id in (("mlp", "CartPole-v1"), ("gru", "CartPole-v1"), ("gru_cont", "Pendulum-v1"), ("mlp_cont", "Pendulum-v1")):
        agent, _ = _agent(kind, env_id)
        _train(agent, 1)
        out = []
        for graphs in (True, False):
            agent.engine.use_graphs = graphs
            out.append([agent.evaluate(64, num_envs=8, seed=4, deterministic=d) for d in (True, False)])   # several chunks
        for g, e in zip(*out):
            assert np.array_equal(g["returns"], e["returns"]) and np.array_equal(g["lengths"], e["lengths"]), kind


def test_custom_network_and_host_environments_evaluate_through_predict():
    from diamond import PPO, PPOConfig, envs
    from diamond.networks import ActorCriticNetwork

    class Custom(ActorCriticNetwork):
        pass
    from diamond.envs import DeviceVectorEnv
    env_fn = DeviceVectorEnv.factory("CartPole-v1", seed=3)
    custom = PPO(env_fn, PPOConfig(num_envs=16, rollout_steps=32, verbose=False, seed=3), network_cls=Custom)
    with torch.no_grad():
        custom.network.actor_head[2].weight.mul_(300.0)
    res = custom.evaluate(8, num_envs=4, seed=3)
    ret, length = _host_loop(custom, env_fn, 4, 8, 3)
    assert np.array_equal(res["returns"], ret) and np.array_equal(res["lengths"], length)
    host = PPO(lambda: envs.CartPoleEnv(), PPOConfig(num_envs=4, rollout_steps=8, verbose=False, seed=3))
    res = host.evaluate(6, num_envs=3, seed=11)
    assert res["lengths"].shape == (6,) and (res["lengths"] >= 1).all() and np.all(res["returns"] == res["lengths"])


# ---- training is not perturbed ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,env_kw", [("mlp", {}), ("gru", {}), ("mlp", dict(normalize_observation=True, normalize_reward=True))])
def test_evaluate_leaves_training_bit_identical(kind, env_kw):
    """k x (rollout + learn), evaluate(), k more == 2k x (rollout + learn): parameters, Adam state, environments and statistics,
    the sampling counter, the numpy and torch streams.  The third rollout (the one that captures the rollout graph) comes after
    evaluate() in the interrupted run."""
    k = 2

    def run(with_eval):
        agent, _ = _agent(kind, "CartPole-v1", seed=13, **env_kw)
        _train(agent, k)
        if with_eval:
            agent.evaluate(10, num_envs=5, seed=99)
            agent.evaluate(4, num_envs=4, deterministic=False)
        for _ in range(k):
            agent.learn(agent.rollout())
        torch.cuda.synchronize()
        eng = agent.engine
        return dict(P=eng.P.clone(), M=eng.M.clone(), V=eng.V.clone(), step=eng.adam_step, draws=eng.draws,
                    envs={n: getattr(agent.envs, n).clone() for n in agent.envs.state_tensors},
                    np=np.random.get_state(legacy=True), torch=torch.get_rng_state().clone(),
                    hx=agent.current_hx.clone() if kind == "gru" else None)

    a, b = run(True), run(False)
    for key in ("P", "M", "V"):
        assert torch.equal(a[key], b[key]), key
    assert a["step"] == b["step"] and a["draws"] == b["draws"]
    for n in a["envs"]:
        assert torch.equal(a["envs"][n], b["envs"][n]), n
    assert a["np"][2] == b["np"][2] and np.array_equal(a["np"][1], b["np"][1])
    assert torch.equal(a["torch"], b["torch"])
    if kind == "gru":
        assert torch.equal(a["hx"], b["hx"])


# ---- learning signal -----------------------------------------------------------------------------------------------------------
# Greedy evaluate(100) after test_cartpole_learns_on_device's training, on one B200 at a 1000 W power limit (tests/evaluate_learning.py):
# seeds 1-5 gave mean lengths 441 / 479 / 371 / 359 / 381 (training-window means 236 / 293 / 280 / 273 / 232).
EVAL_LENGTH_BOUND = 250.0


def test_greedy_policy_after_cartpole_training_balances():
    """test_cartpole_learns_on_device's training, then evaluate(100) of the greedy policy (bound: measured above, with margin)."""
    from diamond import PPO, PPOConfig
    from diamond.envs import DeviceVectorEnv
    cfg = PPOConfig(num_envs=64, rollout_steps=128, verbose=False, seed=1, total_steps=64 * 128 * 40)
    agent = PPO(DeviceVectorEnv.factory("CartPole-v1", seed=1), cfg)
    agent.train()
    res = agent.evaluate(100)
    assert res["lengths"].shape == (100,)
    assert res["mean_length"] > EVAL_LENGTH_BOUND, res["mean_length"]
