"""GPU: the drop-in agents against golden vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py): same initial parameters, same synthetic experience, same
np.random seed -> losses and updated parameters within BASELINE.json's tolerances (1e-4)."""
import glob
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


class Fixture(dict):
    @property
    def files(self):
        return list(self)


def load_fixture(name):
    """learn_<name>.npz merged with learn_<name>.<part>.npz: fixtures that would not fit a file of 1 MB keep the outputs after
    their last epoch in a second file (tests/golden/make_golden.py)."""
    g = Fixture(np.load(os.path.join(GOLDEN, f"learn_{name}.npz")))
    for part in sorted(glob.glob(os.path.join(GOLDEN, f"learn_{name}.*.npz"))):
        g.update(np.load(part))
    return g


def make_env_fn(D, A, cont):
    from diamond import envs
    return lambda: envs.SyntheticEnv(D, A, continuous=cont)


def build_agent(g, epochs, network_cls=None, **extra):
    from diamond import PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig
    D, act, H, N_, T, E, MB, cont = (int(x) for x in g["meta"])
    Agent, Cfg = (ContinuousPPO, ContinuousPPOConfig) if cont else (PPO, PPOConfig)
    cfg = Cfg(num_envs=N_, rollout_steps=T, network_hidden_dim=H, num_epochs=epochs, num_minibatches=MB, verbose=False,
              seed=42, **extra)
    kw = {} if network_cls is None else dict(network_cls=network_cls)
    agent = Agent(make_env_fn(D, act, bool(cont)), cfg, **kw)
    sd = {k[len("init."):]: torch.as_tensor(g[k]) for k in g.files if k.startswith("init.")}
    agent.network.load_state_dict(sd)
    return agent


def experience_from(g):
    T = g["rewards"].shape[0]
    return [[g["obs"][t], g["next_obs"][t], g["actions"][t], g["rewards"][t], g["terminations"][t], g["truncations"][t]]
            for t in range(T)]


def check(agent, g, tag, ptol=1e-4, ltol=1e-4):
    losses = agent.last_losses.cpu().numpy()
    np.testing.assert_allclose(losses, g[f"{tag}.losses"], rtol=ltol, atol=5e-6)
    sd = agent.network.state_dict()
    for k in g.files:
        if k.startswith(f"{tag}.params."):
            name = k[len(f"{tag}.params."):]
            ref = g[k]
            err = np.abs(sd[name].cpu().numpy() - ref).max() / max(np.abs(ref).max(), 1e-12)
            assert err <= ptol, (name, err)


@pytest.mark.parametrize("name", ["C", "L", "Ssmall", "Pn", "Pn3"])
def test_learn_one_epoch_matches_reference(name):
    g = load_fixture(name)
    agent = build_agent(g, 1)
    np.random.seed(123)
    agent.learn(experience_from(g))
    check(agent, g, "e1")
    # the numpy global stream advanced exactly as the reference's np.random.permutation call would have
    B = g["rewards"].size
    after = np.random.randint(0, 2 ** 31, 3)
    np.random.seed(123); np.random.permutation(B)
    np.testing.assert_array_equal(after, np.random.randint(0, 2 ** 31, 3))


@pytest.mark.parametrize("name", ["C", "L", "Ssmall", "Pn", "Pn3"])
def test_learn_default_epochs_matches_reference(name):
    g = load_fixture(name)
    E = int(g["meta"][5])
    agent = build_agent(g, E)
    np.random.seed(123)
    agent.learn(experience_from(g))
    check(agent, g, f"e{E}", ptol=2e-4, ltol=2e-4)


# ---- config S through the tensor-core path: the reference's losses / updated parameters at the benchmark's own shapes ----
def _seeded_case(name):
    """Agent + experience of a seeded fixture (inputs regenerated from the seed, tests/golden/seeded.py; the committed file holds the
    outputs of the UNMODIFIED reference on exactly those inputs)."""
    import sys
    sys.path.insert(0, GOLDEN)
    from seeded import seeded_experience, seeded_params, checksum, state_dict_of
    g = load_fixture(name)
    D, act, H, N_, T, E, MB, _ = (int(x) for x in g["meta"])
    seed = int(g["seed"])
    obs, nobs, actions, rew, term, trunc = seeded_experience(seed, T, N_, D, act)
    init = seeded_params(seed + 1, D, H, act)
    assert checksum([obs, nobs, actions, rew, term, trunc] + [init[k] for k in sorted(init)]) == float(g["checksum"]), \
        "seeded inputs differ from the ones the fixture was generated with"
    exp = [[obs[t], nobs[t], actions[t], rew[t], term[t], trunc[t]] for t in range(T)]
    return g, exp, {k: torch.as_tensor(v) for k, v in state_dict_of(init).items()}, (D, act, H, N_, T, E, MB)


@pytest.mark.parametrize("name,epochs", [("Smid", 1), ("Smid", 4), ("S", 1), ("S", 4)])
def test_learn_config_S_tensor_core_path_matches_reference(name, epochs):
    """north_star's criterion on the named configuration: losses and all 12 updated parameter tensors after one epoch (8 Adam steps,
    where g / sqrt(v) amplifies rounding, SURVEY 0.6) within 1e-4 of the reference (ppo.py:224-287), with every GEMM of the update on
    the 3xTF32 tcgen05 kernels (H = 256, minibatches of 4096 / 65536 rows).  Four epochs: 2e-4, like the small fixtures."""
    from diamond import PPO, PPOConfig
    g, exp, sd, (D, act, H, N_, T, E, MB) = _seeded_case(name)
    cfg = PPOConfig(num_envs=N_, rollout_steps=T, network_hidden_dim=H, num_epochs=epochs, num_minibatches=MB, verbose=False, seed=42)
    agent = PPO(make_env_fn(D, act, False), cfg)
    agent.network.load_state_dict(sd)
    agent.ctx.set_option("tensor_cores", 1)
    l0 = agent.ctx.launches
    np.random.seed(123)
    agent.learn(exp)
    torch.cuda.synchronize()
    tol = 1e-4 if epochs == 1 else 2e-4
    check(agent, g, f"e{epochs}", ptol=tol, ltol=tol)
    # the advantages feeding the update (thin slice kept in the fixture), 1e-5 normalised
    if epochs == 1:
        adv = agent.engine._bufs[(T, N_, epochs, MB, False)]["adv"][:, :16].cpu().numpy()
        ref = g["gae.advantages16"]
        assert np.abs(adv - ref).max() / np.abs(ref).max() <= 1e-5
    assert agent.ctx.launches > l0


def test_learn_config_S_second_learn_replays_graph_and_stays_on_reference():
    """The CUDA-graph replay of the optimiser steps (taken from the second consecutive learn() on the same buffers) gives the same
    update as the eager launches that produced the parity above: two agents, one with graphs disabled, stay bit-identical."""
    from diamond import PPO, PPOConfig
    from diamond.agents import RolloutBuffer
    g, exp, sd, (D, act, H, N_, T, E, MB) = _seeded_case("Smid")
    outs = []
    for use_graphs in (True, False):
        cfg = PPOConfig(num_envs=N_, rollout_steps=T, network_hidden_dim=H, num_epochs=1, num_minibatches=MB, verbose=False, seed=42)
        agent = PPO(make_env_fn(D, act, False), cfg)
        agent.network.load_state_dict(sd)
        agent.engine.use_graphs = use_graphs
        buf = RolloutBuffer.from_lists(agent.ctx, exp, False, agent.device)
        np.random.seed(123)
        for _ in range(3):
            agent.learn(buf)
        torch.cuda.synchronize()
        outs.append((agent.engine.P.clone(), agent.last_losses.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_learn_nondefault_hyperparameters_and_lr_decay():
    g = np.load(os.path.join(GOLDEN, "learn_Cdecay.npz"))
    extra = dict(decay_lr=True, total_steps=8 * 32 * 10, advantage_norm=False, ppo_clip=0.1, value_loss_weight=0.5,
                 entropy_beta=0.02, grad_norm_clip=0.3, gamma=0.97, gae_lambda=0.9)
    agent = build_agent(g, 1, **extra)
    np.random.seed(123)
    agent.learn(experience_from(g))
    check(agent, g, "e1")
    assert abs(agent.optimizer.param_groups[0]["lr"] - float(g["e1.lr_after"])) < 1e-12


def test_adam_state_visible_through_optimizer_state_dict():
    g = np.load(os.path.join(GOLDEN, "learn_C.npz"))
    agent = build_agent(g, 1)
    np.random.seed(123)
    agent.learn(experience_from(g))
    names = [n for n, _ in agent.network.named_parameters()]
    st = agent.optimizer.state_dict()["state"]
    for i, n in enumerate(names):
        np.testing.assert_allclose(st[i]["exp_avg"].cpu().numpy(), g[f"e1.exp_avg.{n}"], rtol=1e-3, atol=1e-7)
        np.testing.assert_allclose(st[i]["exp_avg_sq"].cpu().numpy(), g[f"e1.exp_avg_sq.{n}"], rtol=1e-3, atol=1e-10)
        assert float(st[i]["step"]) == float(g[f"e1.step.{n}"])


def test_calculate_advantage_api_matches_reference():
    g = np.load(os.path.join(GOLDEN, "learn_C.npz"))
    agent = build_agent(g, 1)
    f = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float32))
    adv = agent.calculate_advantage(f(g["rewards"]), f(g["terminations"]), f(g["truncations"]), f(g["gae.values"]),
                                    f(g["gae.next_values"]))
    assert adv.shape == (128, 8) and adv.is_cuda
    ref = g["gae.advantages"]
    assert np.abs(adv.cpu().numpy() - ref).max() / np.abs(ref).max() <= 1e-5


class CustomDiscreteNet(torch.nn.Module):
    """A user network in the style of readme.md:93-109 (different activation, separate trunks)."""

    def __init__(self, observation_space, action_space, cfg):
        super().__init__()
        d, h = int(np.prod(observation_space.shape)), cfg.network_hidden_dim
        self.actor = torch.nn.Sequential(torch.nn.Linear(d, h), torch.nn.ReLU(), torch.nn.Linear(h, action_space.n))
        self.critic = torch.nn.Sequential(torch.nn.Linear(d, h), torch.nn.ReLU(), torch.nn.Linear(h, 1))
        self.actor_out_layer = self.actor[-1]

    def get_actions(self, observations, device):
        with torch.inference_mode():
            logits = self.actor(torch.as_tensor(observations, dtype=torch.float32, device=device))
        return torch.distributions.Categorical(logits=logits).sample().cpu().numpy()

    def get_values(self, observations):
        with torch.inference_mode():
            return self.critic(observations).squeeze(-1)

    def get_logits_and_values(self, x):
        return self.actor(x), self.critic(x).squeeze(-1)


def test_custom_network_path_matches_torch_reference_math():
    """Custom network_cls: kernels for buffer/GAE/gather/loss/clip+Adam around torch autograd.  Checked
    against the same update written with torch ops (the reference's learn() loop, ppo.py:258-285)."""
    from diamond import PPO, PPOConfig, envs
    from oracle import ppo_oracle as O
    D, A, N_, T, MB = 6, 3, 8, 32, 4
    cfg = PPOConfig(num_envs=N_, rollout_steps=T, num_epochs=2, num_minibatches=MB, verbose=False, network_hidden_dim=32)
    agent = PPO(lambda: envs.SyntheticEnv(D, A), cfg, network_cls=CustomDiscreteNet)
    ref_net = CustomDiscreteNet(envs.Box(shape=(D,)), envs.Discrete(A), cfg)
    ref_net.load_state_dict({k: v.detach().cpu().clone() for k, v in agent.network.state_dict().items()})
    rng = np.random.default_rng(0)
    exp = [[rng.standard_normal((N_, D)).astype(np.float32), rng.standard_normal((N_, D)).astype(np.float32),
            rng.integers(0, A, N_), rng.standard_normal(N_), rng.random(N_) < 0.05, rng.random(N_) < 0.05] for _ in range(T)]
    np.random.seed(7)
    agent.learn(exp)
    # torch reference
    obs, nobs, act, rew, term, trunc = (np.asarray(x) for x in zip(*exp))
    t = torch.as_tensor
    obs_t, nobs_t = t(obs), t(nobs)
    with torch.no_grad():
        logits, values = ref_net.get_logits_and_values(obs_t)
        old_lp = torch.distributions.Categorical(logits=logits).log_prob(t(act))
        nv = ref_net.get_values(nobs_t)
    adv = O.gae(rew.astype(np.float32), term.astype(np.float32), trunc.astype(np.float32), values.numpy(), nv.numpy())
    ret, adv_n = O.returns_and_normalise(values.numpy(), adv, True)
    B = T * N_
    opt = torch.optim.Adam(ref_net.parameters(), lr=cfg.lr, eps=cfg.adam_eps)
    np.random.seed(7)
    perms = np.stack([np.random.permutation(B) for _ in range(2)]).reshape(2, MB, B // MB)
    fo, fa, fl, fadv, fret = obs_t.reshape(B, D), t(act).reshape(B), old_lp.reshape(B), t(adv_n).reshape(B), t(ret).reshape(B)
    ref_losses = []
    for pe in perms:
        for mb in pe:
            lg, v = ref_net.get_logits_and_values(fo[mb])
            dist = torch.distributions.Categorical(logits=lg)
            ratio = (dist.log_prob(fa[mb]) - fl[mb]).exp()
            lp = torch.max(-fadv[mb] * ratio, -fadv[mb] * torch.clamp(ratio, 0.8, 1.2)).mean()
            lv = 0.5 * torch.nn.functional.mse_loss(v, fret[mb])
            loss = lp + lv - 0.01 * dist.entropy().mean()
            opt.zero_grad(); loss.backward()
            torch.nn.utils.clip_grad_norm_(ref_net.parameters(), cfg.grad_norm_clip)
            opt.step()
            ref_losses.append(float(loss))
    np.testing.assert_allclose(agent.last_losses[:, 3].cpu().numpy(), ref_losses, rtol=1e-4, atol=1e-6)
    for (n, p), (_, q) in zip(agent.network.named_parameters(), ref_net.named_parameters()):
        err = (p.detach().cpu() - q.detach()).abs().max() / q.detach().abs().max()
        assert float(err) <= 1e-4, (n, float(err))


@pytest.mark.parametrize("env_id,agent_kind", [("CartPole-v1", "ppo"), ("LunarLander-v3", "ppo"), ("Pendulum-v1", "cont")])
def test_train_end_to_end_small(env_id, agent_kind):
    """BASELINE.json configs 1-3 plumbing: agent.train() with rollout -> device buffer -> learn."""
    from diamond import PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig, envs
    if agent_kind == "ppo":
        cfg = PPOConfig(num_envs=8, rollout_steps=128, total_steps=8 * 128 * 3, verbose=False)
        agent = PPO(lambda: envs.make(env_id), cfg)
    else:
        cfg = ContinuousPPOConfig(num_envs=16, rollout_steps=64, total_steps=16 * 64 * 3, verbose=False)
        agent = ContinuousPPO(lambda: envs.make(env_id), cfg)
    before = {k: v.detach().clone() for k, v in agent.network.state_dict().items()}
    agent.train()
    after = agent.network.state_dict()
    assert any(not torch.equal(before[k], after[k]) for k in before)
    assert all(torch.isfinite(v).all() for v in after.values())
    assert torch.isfinite(agent.last_losses).all()
    assert agent.ticker.logs["total_steps"] == cfg.total_steps
    assert agent.engine.adam_step == 3 * cfg.num_epochs * cfg.num_minibatches


def test_cartpole_learns():
    """PPO on CartPole-v1 through the kernels actually improves the policy (mean return > random's ~22)."""
    from diamond import PPO, PPOConfig, envs
    cfg = PPOConfig(num_envs=8, rollout_steps=128, total_steps=8 * 128 * 40, verbose=False)
    agent = PPO(lambda: envs.make("CartPole-v1"), cfg)
    agent.train()
    assert np.mean(agent.ticker.logs["episode_returns"][-20:]) > 60.0


def test_rollout_buffer_matches_reference_list_semantics():
    from diamond import PPO, PPOConfig, envs
    cfg = PPOConfig(num_envs=4, rollout_steps=16, total_steps=64, verbose=False)
    agent = PPO(lambda: envs.make("CartPole-v1"), cfg)
    agent.current_observations, _ = agent.envs.reset(seed=0)
    exp = agent.rollout()
    assert len(exp) == 16
    step = exp[3]
    assert [a.dtype for a in step] == [np.float32, np.float32, np.int64, np.float64, np.bool_, np.bool_]
    assert step[0].shape == (4, 4) and step[2].shape == (4,)
    # obs[t+1] equals next_obs[t] wherever the env was not reset (autoreset disabled semantics)
    for t in range(15):
        done = exp[t][4] | exp[t][5]
        np.testing.assert_array_equal(exp[t + 1][0][~done], exp[t][1][~done])


def test_checkpoint_roundtrip(tmp_path):
    from diamond import PPO, PPOConfig, envs
    from diamond.utils import Checkpointer
    g = np.load(os.path.join(GOLDEN, "learn_C.npz"))
    agent = build_agent(g, 1)
    np.random.seed(123)
    agent.learn(experience_from(g))
    ck = Checkpointer(folder=tmp_path, run_name="t")
    path = ck.save(1024, agent.network, agent.optimizer)
    payload = torch.load(path, map_location="cpu")
    assert set(payload) == {"step", "model_state", "opt_state"}
    agent2 = build_agent(g, 1)
    ck.load(path, agent2.network, agent2.optimizer)
    for k, v in agent.network.state_dict().items():
        assert torch.equal(v, agent2.network.state_dict()[k])
    # resumed agent continues identically (Adam moments restored into the flat buffers)
    np.random.seed(5); agent.learn(experience_from(g))
    np.random.seed(5); agent2.learn(experience_from(g))
    for k, v in agent.network.state_dict().items():
        assert torch.allclose(v, agent2.network.state_dict()[k], rtol=0, atol=0), k


def _recurrent_agent_and_experience(name, network_cls=None):
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    g = np.load(os.path.join(GOLDEN, f"learn_{name}.npz"))
    D, A, H, Hg, N_, T, E, MB = (int(x) for x in g["meta"])
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, num_epochs=E, num_minibatches=MB, verbose=False,
                             network_hidden_dim=H, gru_hidden_dim=Hg, seed=42)
    kw = {} if network_cls is None else dict(network_cls=network_cls)
    agent = RecurrentPPO(lambda: envs.SyntheticEnv(D, A), cfg, **kw)
    sd = {k[len("init."):]: torch.as_tensor(g[k]) for k in g.files if k.startswith("init.")}
    agent.network.load_state_dict(sd)
    hx0 = torch.as_tensor(g["hx0"])
    exp = [[torch.as_tensor(g["obs"][t]), torch.as_tensor(g["actions"][t]), g["rewards"][t], g["terminations"][t], g["truncations"][t],
            torch.as_tensor(g["prev_dones"][t]), torch.as_tensor(g["log_probs"][t]), torch.as_tensor(g["values"][t]),
            torch.as_tensor(g["next_values"][t]), hx0] for t in range(T)]
    return agent, exp, g, E, MB


@pytest.mark.parametrize("name", ["R", "R4", "Rg", "Rw"])
def test_recurrent_learn_matches_reference(name):
    """RecurrentPPO.learn() on the fused recurrent kernels (csrc/rnn.cu) vs the reference (+ the documented 2-line `is None`
    fix, SURVEY §0.4) on recorded rollouts: full-sequence BPTT per minibatch (recurrent_ppo.py:301-367).  R: default sizes,
    one minibatch; R4: four minibatches (row gather / gradient scatter around the scan); Rg: GRU width 24 (shared-memory scan
    kernels); Rw: GRU width 32, 128-wide layers."""
    from diamond.recurrent import FusedRecurrentEngine
    agent, exp, g, E, MB = _recurrent_agent_and_experience(name)
    assert isinstance(agent.engine, FusedRecurrentEngine)
    np.random.seed(123)
    agent.learn(exp)
    check(agent, g, f"e{E}")
    # state_dict / optimizer state keep working (Checkpointer payload, utils.py:584-600)
    st = agent.optimizer.state_dict()["state"]
    assert len(st) == len(list(agent.network.parameters())) and all(float(v["step"]) == E * MB for v in st.values())


def test_recurrent_custom_network_runs_under_autograd_and_matches_reference():
    """A user-supplied network_cls (here: a subclass of the default) is run under torch autograd, with GAE, permutation, loss,
    clip and Adam on the libdppo kernels (RecurrentEngine)."""
    from diamond.recurrent import RecurrentActorCriticNetwork, RecurrentEngine

    class MyNet(RecurrentActorCriticNetwork):
        pass

    agent, exp, g, E, MB = _recurrent_agent_and_experience("R4", network_cls=MyNet)
    assert isinstance(agent.engine, RecurrentEngine)
    np.random.seed(123)
    agent.learn(exp)
    check(agent, g, f"e{E}")


@pytest.mark.parametrize("Hg", [16, 24, 64])
def test_rnn_forward_matches_torch_module(Hg):
    """dppo_rnn_forward (base layer, input projection, forward scan with done-masked resets, heads) vs the torch module the
    reference would run (stepwise nn.GRU semantics are pinned by tests/test_oracle.py::test_recurrent_core_matches_stepwise_nn_gru)."""
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    D, A, H, N_, T = 5, 3, 64, 37, 19
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, network_hidden_dim=H, gru_hidden_dim=Hg, seed=3)
    agent = RecurrentPPO(lambda: envs.SyntheticEnv(D, A), cfg)
    gen = torch.Generator().manual_seed(Hg)
    obs = torch.randn(T, N_, D, generator=gen).cuda()
    dones = (torch.rand(T, N_, generator=gen) < 0.15).cuda()
    hx0 = torch.randn(1, N_, Hg, generator=gen).cuda()
    with torch.no_grad():
        ref_logits, ref_values, ref_hx = agent.network.get_logits_values_and_hx(obs, hx0.clone(), dones)
    logits, values, hx = agent.engine.forward(obs, hx0, dones)
    for got, ref in ((logits, ref_logits), (values, ref_values), (hx, ref_hx)):
        assert (got - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item())
    # no resets, zero initial state, critic only (get_values with dones=None, recurrent_ppo.py:127-136)
    with torch.no_grad():
        ref_v = agent.network.get_values(obs, None, None)
    _, v, _ = agent.engine.forward(obs, None, None, heads=2)
    assert (v - ref_v).abs().max().item() <= 1e-5 * max(1.0, ref_v.abs().max().item())


@pytest.mark.parametrize("Hg,N_,T", [(64, 37, 19), (48, 8, 33), (128, 5, 12), (20, 70, 9), (64, 4099, 4), (64, 1801, 3)])
def test_recurrent_fused_engine_matches_autograd_engine_at_wide_gru(Hg, N_, T):
    """GRU widths beyond the warp kernels (tiled scan kernels; 4 / 2 environments per thread at 4099 / 1801 environments, one
    otherwise; ragged environment counts):
    one learn() of the fused engine equals the same network run under torch autograd (RecurrentEngine) on the same rollout."""
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    from diamond.recurrent import RecurrentActorCriticNetwork, RecurrentRollout, FusedRecurrentEngine, RecurrentEngine

    class Same(RecurrentActorCriticNetwork):
        pass

    D, A, H = 6, 3, 64
    agents = []
    for cls in (RecurrentActorCriticNetwork, Same):
        cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, num_epochs=2, num_minibatches=1, verbose=False, network_hidden_dim=H,
                                 gru_hidden_dim=Hg, seed=4, total_steps=N_ * T * 100)
        agents.append(RecurrentPPO(lambda: envs.SyntheticEnv(D, A), cfg, network_cls=cls))
    fused, auto = agents
    assert isinstance(fused.engine, FusedRecurrentEngine) and isinstance(auto.engine, RecurrentEngine)
    auto.network.load_state_dict(fused.network.state_dict())
    dev = fused.device
    gen = torch.Generator(device=dev).manual_seed(Hg)
    ro = RecurrentRollout(T, N_, D, Hg, dev)
    ro.obs.normal_(generator=gen); ro.actions.random_(0, A, generator=gen); ro.rewards.normal_(generator=gen)
    ro.terminations.copy_((torch.rand(T, N_, device=dev, generator=gen) < 0.1).float()); ro.truncations.zero_()
    ro.prev_dones.copy_(torch.rand(T, N_, device=dev, generator=gen) < 0.1)
    ro.log_probs.fill_(-float(np.log(A))); ro.values.normal_(generator=gen); ro.next_values.normal_(generator=gen)
    ro.hx0.normal_(generator=gen); ro.filled = T
    for ag in (fused, auto):
        np.random.seed(8)
        ag.learn(ro)
    torch.cuda.synchronize()
    for (k, p), (_, q) in zip(fused.network.named_parameters(), auto.network.named_parameters()):
        err = float((p - q).abs().max() / q.abs().max().clamp_min(1e-12))
        assert err <= 1e-4, (k, err)
    assert float((fused.last_losses - auto.last_losses).abs().max()) <= 1e-4


def test_recurrent_train_runs_on_cartpole():
    """Plumbing run of config 4 (RecurrentPPO on CartPole-v1): rollout with done-masked hidden resets, learn, LR schedule."""
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    cfg = RecurrentPPOConfig(num_envs=8, rollout_steps=16, num_epochs=2, num_minibatches=1, total_steps=8 * 16 * 3, verbose=False, seed=1)
    agent = RecurrentPPO(lambda: envs.make("CartPole-v1"), cfg)
    before = {k: v.detach().clone() for k, v in agent.network.state_dict().items()}
    agent.train()
    after = agent.network.state_dict()
    assert any(not torch.equal(before[k], after[k]) for k in before)
    assert all(torch.isfinite(v).all() for v in after.values())
    assert torch.isfinite(agent.last_losses).all()
    ro_like = agent.engine.last_losses.shape
    assert ro_like == (2, 4)


def test_graph_replay_of_update_loop_is_bit_identical_to_eager():
    """From the second consecutive learn() on the same device buffer the optimiser steps of an epoch are replayed as a CUDA
    graph (device-resident indices and Adam step constants); parameters, Adam state and losses must equal the eager path
    bit for bit, and the numpy stream must advance identically."""
    from diamond import PPO, PPOConfig, envs
    from diamond.agents import RolloutBuffer
    D, A, H, N_, T = 16, 4, 256, 64, 64                      # 4096 rows, minibatches of 1024: tensor-core path
    rng = np.random.default_rng(3)
    exp = [[rng.standard_normal((N_, D)).astype(np.float32), rng.standard_normal((N_, D)).astype(np.float32),
            rng.integers(0, A, N_), rng.standard_normal(N_), rng.random(N_) < 0.05, rng.random(N_) < 0.05] for _ in range(T)]

    def run(use_graphs):
        cfg = PPOConfig(num_envs=N_, rollout_steps=T, network_hidden_dim=H, num_epochs=3, num_minibatches=4, verbose=False, seed=7,
                        total_steps=N_ * T * 10)
        agent = PPO(lambda: envs.SyntheticEnv(D, A), cfg)
        agent.engine.use_graphs = use_graphs
        buf = RolloutBuffer.from_lists(agent.ctx, exp, False, agent.device)
        np.random.seed(99)
        all_losses = []
        for _ in range(3):
            agent.learn(buf)
            all_losses.append(agent.last_losses.clone())
        torch.cuda.synchronize()
        return agent, torch.cat(all_losses), np.random.randint(0, 2 ** 31, 2)

    a0, l0, r0 = run(False)
    a1, l1, r1 = run(True)
    assert a1.engine._bufs and any(b.get("graph") for b in a1.engine._bufs.values()), "graph path was not taken"
    assert torch.equal(l0, l1)
    assert torch.equal(a0.engine.P, a1.engine.P) and torch.equal(a0.engine.M, a1.engine.M) and torch.equal(a0.engine.V, a1.engine.V)
    assert a0.engine.adam_step == a1.engine.adam_step == 3 * 3 * 4
    np.testing.assert_array_equal(r0, r1)


@pytest.mark.parametrize("kind", ["device", "host"])
def test_train_resume_is_bit_identical_to_uninterrupted_run(tmp_path, kind):
    """SURVEY 8 f3: train(resume_from=checkpoint) restores model, Adam moments + step, LinearLR, the numpy / counter-based RNG streams,
    the environments and the Ticker; an interrupted + resumed run ends with bit-identical parameters, optimiser state and episode
    statistics.  (The reference saves checkpoints, ppo.py:303-310 / utils.py:584-600, but never loads them.)"""
    from diamond import PPO, PPOConfig, envs
    from diamond.envs import DeviceVectorEnv
    from diamond.utils import Checkpointer
    N_, T, R = (64, 32, 7) if kind == "device" else (4, 16, 6)

    def make(tag):
        cfg = PPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=5, total_steps=N_ * T * R, decay_lr=True, num_minibatches=4)
        env_fn = DeviceVectorEnv.factory("CartPole-v1", seed=5) if kind == "device" else (lambda: envs.CartPoleEnv())
        agent = PPO(env_fn, cfg)
        agent.checkpointer = Checkpointer(tmp_path / tag, "run")
        return agent

    full = make("full")
    full.train()
    part = make("part")
    part.train(max_rollouts=3)
    path = part.last_checkpoint
    chk = torch.load(path, map_location="cpu", weights_only=False)
    assert {"step", "model_state", "opt_state", "train_state"} <= set(chk) and chk["step"] == 3 * N_ * T     # reference payload keys kept
    resumed = make("resumed")
    resumed.train(resume_from=path)
    torch.cuda.synchronize()
    assert torch.equal(resumed.engine.P, full.engine.P)
    assert torch.equal(resumed.engine.M, full.engine.M) and torch.equal(resumed.engine.V, full.engine.V)
    assert resumed.engine.adam_step == full.engine.adam_step == R * 4 * 4
    assert resumed.optimizer.param_groups[0]["lr"] == full.optimizer.param_groups[0]["lr"]
    a, b = resumed.ticker.logs, full.ticker.logs
    for k in ("total_steps", "total_episodes", "episode_returns", "episode_lengths"):
        assert a[k] == b[k], k
    # and the interrupted agent itself was not at the end
    assert not torch.equal(part.engine.P, full.engine.P)


@pytest.mark.parametrize("cont,D,A,N_,T,MB", [(False, 4, 2, 8, 128, 8), (False, 8, 4, 5, 20, 1), (True, 3, 1, 64, 64, 8), (True, 5, 3, 7, 33, 3),
                                              (False, 30, 8, 16, 64, 2), (False, 17, 5, 4, 100, 4),
                                              (False, 4, 2, 64, 128, 8), (True, 6, 3, 64, 128, 8), (False, 5, 3, 37, 40, 2), (True, 3, 2, 37, 40, 2)])
def test_small_net_cluster_kernel_matches_per_layer_kernels(cont, D, A, N_, T, MB):
    """Default 64-wide networks: the one-launch cluster kernel (dppo_small_update: whole update loop in distributed shared memory)
    against the per-layer kernel path on the same learn(): losses and parameters agree to fp32 summation order, Adam moments too.
    Ragged shapes: rows per minibatch that are not multiples of the 16-row tile or of the 8 CTAs.  1024 rows (the SMALL_ROWS bound)
    and 740 rows give each CTA two tiles, full and ragged.  D = 30 is the largest obs_dim the kernel takes with 8 actions."""
    from diamond import PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig, envs
    Agent, Cfg = (ContinuousPPO, ContinuousPPOConfig) if cont else (PPO, PPOConfig)
    rng = np.random.default_rng(D * 7 + A)
    exp = [[rng.standard_normal((N_, D)).astype(np.float32), rng.standard_normal((N_, D)).astype(np.float32),
            rng.standard_normal((N_, A)).astype(np.float32) if cont else rng.integers(0, A, N_), rng.standard_normal(N_),
            rng.random(N_) < 0.05, rng.random(N_) < 0.05] for _ in range(T)]
    outs = []
    for small in (True, False):
        cfg = Cfg(num_envs=N_, rollout_steps=T, num_epochs=3, num_minibatches=MB, verbose=False, seed=11)
        agent = Agent(lambda: envs.SyntheticEnv(D, A, continuous=cont), cfg)
        agent.engine.use_small_kernel = small
        np.random.seed(5)
        agent.learn(exp)
        agent.learn(exp)                                   # Adam moments / step carried into a second launch
        torch.cuda.synchronize()
        assert any("small" in b for b in agent.engine._bufs.values()) == small       # the cluster kernel ran exactly when enabled
        outs.append((agent.engine.P.clone(), agent.engine.M.clone(), agent.engine.V.clone(), agent.last_losses.clone(), agent.engine.adam_step))
    (p1, m1, v1, l1, s1), (p0, m0, v0, l0, s0) = outs
    assert s1 == s0 == 2 * 3 * MB
    np.testing.assert_allclose(l1.cpu().numpy(), l0.cpu().numpy(), rtol=2e-5, atol=2e-6)
    assert float((p1 - p0).abs().max() / p0.abs().max()) <= 2e-5
    assert float((m1 - m0).abs().max()) <= 1e-5 * max(1.0, float(m0.abs().max()))
    assert float((v1 - v0).abs().max()) <= 1e-5 * max(1e-3, float(v0.abs().max()))


def test_recurrent_graph_replay_is_bit_identical_to_eager():
    """RecurrentPPO.learn(): from the second call on the same rollout tensors the optimiser steps (15 launches each) are replayed as a
    CUDA graph with device-resident step constants; parameters and losses equal the eager launches bit for bit."""
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    from diamond.recurrent import RecurrentRollout
    g = np.load(os.path.join(GOLDEN, "learn_R4.npz"))
    D, A, H, Hg, N_, T, E, MB = (int(x) for x in g["meta"])
    outs = []
    for use_graphs in (True, False):
        cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, num_epochs=E, num_minibatches=MB, verbose=False, network_hidden_dim=H,
                                 gru_hidden_dim=Hg, seed=2)
        agent = RecurrentPPO(lambda: envs.SyntheticEnv(D, A), cfg)
        agent.network.load_state_dict({k[len("init."):]: torch.as_tensor(g[k]) for k in g.files if k.startswith("init.")})
        agent.engine.use_graphs = use_graphs
        ro = RecurrentRollout(T, N_, D, Hg, agent.device)
        for name in ("obs", "actions", "rewards", "terminations", "truncations", "prev_dones", "log_probs", "values", "next_values"):
            getattr(ro, name).copy_(torch.as_tensor(g[name]).to(getattr(ro, name).dtype))
        ro.hx0.copy_(torch.as_tensor(g["hx0"]).reshape(ro.hx0.shape))
        ro.filled = T
        np.random.seed(123)
        for _ in range(3):
            agent.learn(ro)
        torch.cuda.synchronize()
        outs.append((agent.engine.P.clone(), agent.last_losses.clone()))
        if use_graphs:
            assert any(b["graphs"] for b in agent.engine._bufs.values()), "graph path was not taken"
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_recurrent_device_rollout_matches_module_and_learns():
    """RecurrentPPO on device-resident CartPole: the rollout recorded on the device (GRU step, sampling, environment kernel, V(final
    obs | h_{t+1})) is what the torch module computes from the same observations / hidden states / resets (recurrent_ppo.py:214-263),
    prev_dones chain the environment's done flags, and train() improves the policy."""
    from diamond import RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    N_, T = 32, 32
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=4, total_steps=N_ * T * 60)
    agent = RecurrentPPO(DeviceVectorEnv.factory("CartPole-v1", seed=4), cfg)
    agent.current_observations, _ = agent.envs.reset(seed=4)
    agent.prev_dones = np.zeros(N_, dtype=bool)
    agent.current_hx = torch.zeros(1, N_, cfg.gru_hidden_dim, device=agent.device)
    ro = agent.rollout()
    torch.cuda.synchronize()
    dones = (ro.terminations + ro.truncations) > 0
    assert torch.equal(ro.prev_dones[1:], dones[:-1]) and not ro.prev_dones[0].any()
    assert torch.all(ro.rewards == 1.0) and dones.any()
    # the torch module on the recorded sequence reproduces the recorded values and log-probs
    with torch.inference_mode():
        logits, values, _ = agent.network.get_logits_values_and_hx(ro.obs, ro.hx0.clone(), ro.prev_dones)
    lp = torch.distributions.Categorical(logits=logits).log_prob(ro.actions)
    assert float((values - ro.values).abs().max()) <= 1e-5 and float((lp - ro.log_probs).abs().max()) <= 1e-5
    assert bool(torch.isfinite(ro.next_values).all())
    agent.train()
    lengths = agent.ticker.logs["episode_lengths"]
    assert len(lengths) > 10 and np.mean(lengths) > 40.0, np.mean(lengths)


def test_recurrent_rollout_graph_replay_is_bit_identical_to_eager():
    """The recurrent device rollout replayed as one CUDA graph (from the third rollout; draw counters relative to a device-resident
    base) records exactly what the eager launches record."""
    from diamond import RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    N_, T = 48, 17                                           # odd T: the hidden-state ping-pong ends in the other buffer
    recs = []
    for use_graphs in (True, False):
        cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=6, total_steps=N_ * T * 100)
        agent = RecurrentPPO(DeviceVectorEnv.factory("CartPole-v1", seed=6), cfg)
        agent.engine.use_graphs = use_graphs
        agent.ticker = None
        agent.current_observations, _ = agent.envs.reset(seed=6)
        agent.prev_dones = np.zeros(N_, dtype=bool)
        agent.current_hx = torch.zeros(1, N_, cfg.gru_hidden_dim, device=agent.device)
        out = []
        for _ in range(5):
            ro = agent.rollout()
            out.append([getattr(ro, k).clone() for k in ("obs", "actions", "rewards", "terminations", "truncations", "prev_dones", "log_probs",
                                                         "values", "next_values", "hx0")])
        torch.cuda.synchronize()
        if use_graphs:
            assert agent._ro_graph is not None, "graph path was not taken"
        recs.append(out)
    for a, b in zip(*recs):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
