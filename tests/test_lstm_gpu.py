"""LSTM networks (dppo_rnn_desc.cell = 1) on the GPU: the fused LSTM scans through the C ABI against a float64 CPU autograd
reference on every scan instantiation, and RecurrentPPO / RecurrentContinuousPPO with the LSTM networks.

The reference is RecurrentLSTMActorCriticNetwork / RecurrentContinuousLSTMActorCriticNetwork in float64 on the CPU, loaded from the
same flat fp32 parameter buffer, with the PPO losses of test_rnn_kernels_gpu.py (categorical) and test_rnn_gaussian_gpu.py
(Gaussian).  The case table and the mirror of the branch choice are in test_lstm.py, which checks them on the CPU."""
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_lstm import CASES, CASE_IDS, lstm_branch
from test_rnn_kernels_gpu import GRAD_TOL, cuda, make_hyper, nerr
from test_rnn_kernels_gpu import reference_loss as discrete_loss, set_old_log_probs
from test_rnn_gaussian_gpu import reference_loss as gaussian_loss, set_actions_and_old_log_probs

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------- inputs and the float64 reference -----------------------------
def make_inputs(case, seed=0):
    cid, br, D, H, Hg, A, T, N, opts = case
    rng = np.random.default_rng(1000 * CASE_IDS.index(cid) + seed + 777)
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    gauss = "gauss" in opts
    desc = Nt.RnnDesc(D, H, Hg, A, int(gauss), 1)
    lay = Nt.rnn_layout(desc)
    slices = rnn_param_slices(desc, lay)
    flat = np.zeros(int(lay.total), np.float32)
    for name, (off, shape) in slices.items():
        if name == "actor_log_std":
            w = rng.uniform(-1.0, 0.3, shape)
        elif len(shape) == 2:
            w = rng.standard_normal(shape) / np.sqrt(shape[1])
        else:
            w = 0.3 * rng.standard_normal(shape)
        flat[off:off + int(np.prod(shape))] = w.reshape(-1)
    obs = rng.standard_normal((T, N, D)).astype(np.float32)
    hx0 = (0.5 * rng.standard_normal((N, 2 * Hg))).astype(np.float32) if "hx0" in opts else None     # h0 | c0
    dones = None
    if "dones" in opts:
        dones = rng.random((T, N)) < 0.15
        dones[np.arange(T), rng.integers(0, N, T)] = True
        dones[0, : max(1, N // 3)] = True
    actions = rng.integers(0, A, (T, N)).astype(np.int32)
    adv = rng.standard_normal((T, N)).astype(np.float32)
    ret = rng.standard_normal((T, N)).astype(np.float32)
    return SimpleNamespace(case=case, desc=desc, lay=lay, slices=slices, flat=flat, obs=obs, hx0=hx0, dones=dones, actions=actions,
                           adv=adv, ret=ret, rng=rng, D=D, H=H, Hg=Hg, A=A, T=T, N=N, gauss=gauss)


def reference_network(x):
    from diamond.config import RecurrentContinuousPPOConfig, RecurrentPPOConfig
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork, RecurrentLSTMActorCriticNetwork
    if x.gauss:
        net = RecurrentContinuousLSTMActorCriticNetwork(SimpleNamespace(shape=(x.D,)), SimpleNamespace(shape=(x.A,)),
                                                        RecurrentContinuousPPOConfig(network_hidden_dim=x.H, gru_hidden_dim=x.Hg))
    else:
        net = RecurrentLSTMActorCriticNetwork(SimpleNamespace(shape=(x.D,)), SimpleNamespace(n=x.A),
                                              RecurrentPPOConfig(network_hidden_dim=x.H, gru_hidden_dim=x.Hg))
    net = net.double()
    params = dict(net.named_parameters())
    assert set(params) == set(x.slices)
    with torch.no_grad():
        for name, (off, shape) in x.slices.items():
            params[name].copy_(torch.as_tensor(x.flat[off:off + int(np.prod(shape))].astype(np.float64)).reshape(shape))
    return net


def reference_forward(x, net, with_state=True):
    """(head [T,N,A] (logits or means), log_std or None, values [T,N], hx [1,N,2Hg])."""
    obs = torch.as_tensor(x.obs, dtype=torch.float64)
    hx = torch.as_tensor(x.hx0, dtype=torch.float64).unsqueeze(0) if (with_state and x.hx0 is not None) else None
    dn = torch.as_tensor(x.dones) if (with_state and x.dones is not None) else None
    if x.gauss:
        return net.get_means_log_stds_values_and_hx(obs, hx, dn)
    logits, values, hx = net.get_logits_values_and_hx(obs, hx, dn)
    return logits, None, values, hx


@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as Nt
    return Nt.get_context(0)


def check_grad_vs_fp64(ctx, case):
    """The flat gradient (every tensor), the four losses and the clip norm, for the whole rollout (idx NULL) and a permutation slice,
    against float64 autograd; padding between the tensors comes out zero."""
    cid, br, D, H, Hg, A, T, N, opts = case
    x = make_inputs(case)
    B = T * N
    net = reference_network(x)
    head, log_std, values, _ = reference_forward(x, net)
    if x.gauss:
        set_actions_and_old_log_probs(x, head, log_std)
        actions = cuda(x.actions.reshape(B, A))
    else:
        lsm = torch.log_softmax(head.detach().reshape(B, A), -1)
        set_old_log_probs(x, lsm.gather(-1, torch.as_tensor(x.actions.reshape(B, 1).astype(np.int64))).squeeze(-1).numpy())
        actions = cuda(x.actions.reshape(B), torch.int32)
    a64 = x.adv.astype(np.float64).reshape(-1)
    P, obs, pd, hx0 = cuda(x.flat), cuda(x.obs), cuda(x.dones, torch.uint8), cuda(x.hx0)
    old_lp, adv, ret = cuda(x.old_lp), cuda(x.adv.reshape(B)), cuda(x.ret.reshape(B))
    stats = cuda(np.array([a64.sum(), (a64 ** 2).sum()]), torch.float64)
    adv_norm = "norm" in opts
    Mp = max(1, 3 * B // 8)
    perm = x.rng.permutation(B).astype(np.int32)
    used = torch.zeros(int(x.lay.total), dtype=torch.bool)
    for off, shape in x.slices.values():
        used[off:off + int(np.prod(shape))] = True
    sumsq = torch.zeros(ctx.grad_sumsq_bytes(int(x.lay.total)) // 8 + 1, dtype=torch.float64, device="cuda")
    adam_ws = torch.empty(ctx.clip_adam_workspace_bytes(int(x.lay.total)) // 8 + 1, dtype=torch.float64, device="cuda")
    for rows, M in ((None, B), (perm[:Mp], Mp)):
        den = 2 * M if "den2" in opts else M
        rsel = np.arange(B) if rows is None else rows.astype(np.int64)
        net.zero_grad()
        if x.gauss:
            total, ref_losses = gaussian_loss(x, head, log_std, values, rsel, adv_norm, den)
        else:
            total, ref_losses = discrete_loss(x, head, values, rsel, adv_norm, den)
        total.backward(retain_graph=True)
        ref = {n: p.grad.numpy() for n, p in net.named_parameters()}
        hyper = make_hyper(M, den, adv_norm, B)
        hyper.grad_sumsq = sumsq.data_ptr()
        ws = torch.empty(ctx.rnn_workspace_bytes(x.desc, T, N, M, True) // 4 + 64, device="cuda")
        grads = torch.full((int(x.lay.total),), 7.0, device="cuda")
        losses = torch.zeros(4, device="cuda")
        ctx.rnn_grad_minibatch(x.desc, P, grads, obs, pd, hx0, T, N, actions, old_lp, adv, ret, stats, cuda(rows, torch.int32), M,
                               hyper, losses, ws)
        torch.cuda.synchronize()
        where = f"{cid} M={M}"
        np.testing.assert_allclose(losses.cpu().numpy(), [float(l) for l in ref_losses], rtol=1e-5, atol=1e-6, err_msg=where)
        g = grads.cpu()
        assert float(g[~used].abs().sum()) == 0.0, where
        for n in x.slices:
            off, shape = x.slices[n]
            got = g[off:off + int(np.prod(shape))].numpy().reshape(ref[n].shape)
            assert nerr(got, ref[n]) <= GRAD_TOL, (where, n, nerr(got, ref[n]))
        ref_norm = float(np.sqrt(sum((r.astype(np.float64) ** 2).sum() for r in ref.values())))
        gn = torch.zeros(1, device="cuda")
        z = torch.zeros_like(grads)
        ctx.clip_adam_step(P.clone(), grads.clone(), z, z.clone(), hyper, adam_ws, gn)
        torch.cuda.synchronize()
        assert abs(float(gn) - ref_norm) <= GRAD_TOL * ref_norm, (where, float(gn), ref_norm)


# ---------------------------------------------------------------- GPU: kernels against float64 --------------------------------
@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_lstm_rnn_grad_minibatch_vs_fp64(ctx, case):
    check_grad_vs_fp64(ctx, case)


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_lstm_rnn_forward_vs_fp64(ctx, case):
    """dppo_rnn_forward with cell = 1, heads 1, 2 and 3, with and without resets / initial state: logits or means, values and the
    packed final state h | c within 1e-5 max(1, |ref|) of float64."""
    cid, br, D, H, Hg, A, T, N, opts = case
    x = make_inputs(case, seed=1)
    net = reference_network(x)
    ws = torch.empty(ctx.rnn_workspace_bytes(x.desc, T, N, T * N, False) // 4 + 64, device="cuda")
    P, obs = cuda(x.flat), cuda(x.obs)
    tol = lambda ref: 1e-5 * max(1.0, float(np.abs(ref).max()))
    for with_state in (True, False):
        with torch.no_grad():
            rl, _, rv, rh = reference_forward(x, net, with_state)
            rl, rv, rh = rl.numpy(), rv.numpy(), rh.numpy()
        pd = cuda(x.dones, torch.uint8) if with_state else None
        hx0 = cuda(x.hx0) if with_state else None
        for heads in (1, 2, 3):
            logits = torch.full((T, N, A), float("nan"), device="cuda") if heads & 1 else None
            values = torch.full((T, N), float("nan"), device="cuda") if heads & 2 else None
            hx = torch.full((N, 2 * Hg), float("nan"), device="cuda")
            ctx.rnn_forward(x.desc, P, obs, pd, hx0, T, N, heads, logits, values, hx, ws)
            torch.cuda.synchronize()
            where = (cid, with_state, heads)
            if heads & 1:
                assert np.abs(logits.cpu().numpy() - rl).max() <= tol(rl), where
            if heads & 2:
                assert np.abs(values.cpu().numpy() - rv).max() <= tol(rv), where
            assert np.abs(hx.cpu().numpy() - rh[0]).max() <= tol(rh), where


def _random_params(desc, seed):
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    lay = Nt.rnn_layout(desc)
    rng = np.random.default_rng(seed)
    flat = np.zeros(int(lay.total), np.float32)
    for name, (off, shape) in rnn_param_slices(desc, lay).items():
        s = 1.0 / np.sqrt(shape[1]) if len(shape) == 2 else 0.3
        flat[off:off + int(np.prod(shape))] = (rng.standard_normal(int(np.prod(shape))) * s).astype(np.float32)
    return cuda(flat), rng


@gpu
@pytest.mark.parametrize("Hg,Ns", [(64, (64, 1801, 4099)), (256, (5, 161, 321)), (128, (20, 331, 621))])
def test_lstm_results_do_not_depend_on_env_count(ctx, Hg, Ns):
    """The same environments inside larger N: tiled E = 1 / 2 / 4 at Hg = 64, cluster E = 1 / 2 / 4 with C = 8 at 256 and C = 4 at
    128 (where the environments also move to other cluster slots).  Logits, values and the packed final state are bit-identical."""
    from diamond import _native as Nt
    D, H, A, T = 8, 64, 4, 8
    desc = Nt.RnnDesc(D, H, Hg, A, 0, 1)
    P, rng = _random_params(desc, Hg)
    Nmax, K = max(Ns), min(Ns)
    obs = rng.standard_normal((T, Nmax, D)).astype(np.float32)
    dones = rng.random((T, Nmax)) < 0.15
    hx0 = (0.5 * rng.standard_normal((Nmax, 2 * Hg))).astype(np.float32)
    out = {}
    branches = set()
    for N in Ns:
        branches.add(lstm_branch(N, Hg))
        ws = torch.empty(ctx.rnn_workspace_bytes(desc, T, N, T * N, False) // 4 + 64, device="cuda")
        logits, values, hx = (torch.empty(T, N, A, device="cuda"), torch.empty(T, N, device="cuda"),
                              torch.empty(N, 2 * Hg, device="cuda"))
        ctx.rnn_forward(desc, P, cuda(obs[:, :N]), cuda(dones[:, :N], torch.uint8), cuda(hx0[:N]), T, N, 3, logits, values, hx, ws)
        torch.cuda.synchronize()
        out[N] = (logits[:, :K].cpu(), values[:, :K].cpu(), hx[:K].cpu())
    assert len(branches) == 3, branches
    for N in Ns[1:]:
        for k, what in enumerate(("logits", "values", "hx_out")):
            assert torch.equal(out[N][k], out[K][k]), (Hg, N, what)


@gpu
@pytest.mark.parametrize("Hg", [4, 10, 98, 260])
def test_lstm_rnn_refusals(ctx, Hg):
    """LSTM widths outside the rule (a multiple of 4 from 8 to 256) are refused by both calls, naming the rule, before anything is
    launched; the context then computes a correct gradient."""
    from diamond import _native as Nt
    D, H, A, T, N = 4, 32, 2, 2, 3
    B = T * N
    desc = Nt.RnnDesc(D, H, Hg, A, 0, 1)
    lay = Nt.rnn_layout(desc)
    P = torch.zeros(int(lay.total), device="cuda")
    ws = torch.empty(1 << 20, device="cuda")
    launches = ctx.launches
    f = lambda *s: torch.zeros(*s, device="cuda")
    with pytest.raises(Nt.NativeError, match="multiple of 4 from 8 to 256"):
        ctx.rnn_forward(desc, P, f(T, N, D), None, None, T, N, 3, f(T, N, A), f(T, N), f(N, 2 * Hg), ws)
    with pytest.raises(Nt.NativeError, match="multiple of 4 from 8 to 256"):
        ctx.rnn_grad_minibatch(desc, P, f(int(lay.total)), f(T, N, D), None, None, T, N, f(B).to(torch.int32), f(B), f(B), f(B), None,
                               None, B, make_hyper(B, B, False, B), f(4), ws)
    assert ctx.launches == launches
    check_grad_vs_fp64(ctx, CASES[CASE_IDS.index("w16")])


# ---------------------------------------------------------------- GPU: agent level ---------------------------------------------
def _synthetic_rollout(T, N_, D, A, S, dev, seed, continuous):
    import math
    from diamond.recurrent import RecurrentRollout
    gen = torch.Generator(device=dev).manual_seed(seed)
    ro = RecurrentRollout(T, N_, D, S, dev, A if continuous else None)
    ro.obs.normal_(generator=gen)
    if continuous:
        ro.actions.normal_(generator=gen)
        ro.log_probs.copy_(-0.5 * (ro.actions ** 2).sum(-1) - 0.5 * A * math.log(2 * math.pi))
    else:
        ro.actions.copy_(torch.randint(0, A, (T, N_), device=dev, generator=gen))
        ro.log_probs.fill_(-math.log(A))
    ro.rewards.normal_(generator=gen)
    ro.terminations.copy_((torch.rand(T, N_, device=dev, generator=gen) < 0.1).float()); ro.truncations.zero_()
    ro.prev_dones.copy_(torch.rand(T, N_, device=dev, generator=gen) < 0.1)
    ro.values.normal_(generator=gen); ro.next_values.normal_(generator=gen)
    ro.hx0.normal_(generator=gen); ro.filled = T
    return ro


@gpu
@pytest.mark.parametrize("continuous", [False, True])
@pytest.mark.parametrize("Hg,N_,T", [(16, 24, 16), (64, 20, 9), (256, 38, 19)])
def test_lstm_fused_engine_matches_autograd_engine(Hg, N_, T, continuous):
    """The fused engine (the LSTM network class itself) equals the same network under torch autograd (RecurrentEngine, selected by a
    subclass) after one learn() of 2 epochs x 2 minibatches on the same rollout: parameters and losses within 2e-5, at the warp (16),
    tiled (64) and cluster (256) widths."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig, RecurrentPPO, RecurrentPPOConfig, envs
    from diamond.recurrent import (FusedRecurrentEngine, RecurrentContinuousLSTMActorCriticNetwork, RecurrentEngine,
                                   RecurrentLSTMActorCriticNetwork)
    Agent, Cfg, Net = ((RecurrentContinuousPPO, RecurrentContinuousPPOConfig, RecurrentContinuousLSTMActorCriticNetwork) if continuous
                       else (RecurrentPPO, RecurrentPPOConfig, RecurrentLSTMActorCriticNetwork))

    class Same(Net):
        pass

    D, A, H = 6, 3, 64
    agents = []
    for cls in (Net, Same):
        cfg = Cfg(num_envs=N_, rollout_steps=T, num_epochs=2, num_minibatches=2, verbose=False, network_hidden_dim=H, gru_hidden_dim=Hg,
                  seed=4, total_steps=N_ * T * 100)
        agents.append(Agent(lambda: envs.SyntheticEnv(D, A, continuous=continuous), cfg, network_cls=cls))
    fused, auto = agents
    assert isinstance(fused.engine, FusedRecurrentEngine) and isinstance(auto.engine, RecurrentEngine)
    assert fused.engine.desc.cell == 1 and fused.state_dim == auto.state_dim == 2 * Hg
    auto.network.load_state_dict(fused.network.state_dict())
    ro = _synthetic_rollout(T, N_, D, A, 2 * Hg, fused.device, Hg, continuous)
    for ag in (fused, auto):
        np.random.seed(8)
        ag.learn(ro)
    torch.cuda.synchronize()
    for (k, p), (_, q) in zip(fused.network.named_parameters(), auto.network.named_parameters()):
        err = float((p - q).abs().max() / q.abs().max().clamp_min(1e-12))
        assert err <= 2e-5, (k, err)
    assert float((fused.last_losses - auto.last_losses).abs().max()) <= 2e-5


def _lstm_agent(kind, env_id, seed=3, num_envs=16, Hg=32, T=32, **kw):
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig, RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork, RecurrentLSTMActorCriticNetwork
    Agent, Cfg, Net = ((RecurrentContinuousPPO, RecurrentContinuousPPOConfig, RecurrentContinuousLSTMActorCriticNetwork)
                       if kind == "cont" else (RecurrentPPO, RecurrentPPOConfig, RecurrentLSTMActorCriticNetwork))
    cfg = Cfg(num_envs=num_envs, rollout_steps=T, verbose=False, seed=seed, total_steps=num_envs * T * 100, gru_hidden_dim=Hg, **kw)
    env_fn = DeviceVectorEnv.factory(env_id, seed=seed)
    return Agent(env_fn, cfg, network_cls=Net), env_fn


def _start(agent):
    n = agent.cfg.num_envs
    agent.current_observations, _ = agent.envs.reset(seed=agent.cfg.seed)
    agent.prev_dones = np.zeros(n, dtype=bool)
    agent.current_hx = torch.zeros(1, n, agent.state_dim, device=agent.device)


@gpu
@pytest.mark.parametrize("kind,env_id", [("disc", "CartPole-v1"), ("cont", "Pendulum-v1")])
def test_lstm_device_rollout_graph_replay_and_module(kind, env_id):
    """Device rollout (odd T, so the state ping-pongs): the CUDA-graph replay records exactly what eager launches record, and the
    recorded values and log-probs are what the float64 module computes from the recorded sequence and packed hx0, to 1e-5."""
    N_, T, Hg = 48, 17, 16
    recs = []
    for use_graphs in (True, False):
        agent, _ = _lstm_agent(kind, env_id, seed=6, num_envs=N_, Hg=Hg, T=T)
        agent.engine.use_graphs = use_graphs
        agent.ticker = None
        _start(agent)
        out = []
        for _ in range(5):
            ro = agent.rollout()
            out.append([getattr(ro, k).clone() for k in ("obs", "actions", "prev_dones", "log_probs", "values", "next_values", "hx0")])
        torch.cuda.synchronize()
        if use_graphs:
            assert agent._ro_graph is not None, "graph path was not taken"
            net64 = agent.network.double().cpu()
        recs.append(out)
    for a, b in zip(*recs):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    assert any(bool(r[6].abs().sum() > 0) for r in recs[0][1:])         # the carried state (h | c) is not zero after a rollout
    for obs, actions, prev_dones, log_probs, values, next_values, hx0 in recs[0]:
        assert hx0.shape == (1, N_, 2 * Hg)
        with torch.inference_mode():
            if kind == "cont":
                mean, ls, v, _ = net64.get_means_log_stds_values_and_hx(obs.double().cpu(), hx0.double().cpu(), prev_dones.cpu())
                lp = torch.distributions.Normal(mean, ls.exp()).log_prob(actions.double().cpu()).sum(-1)
            else:
                logits, v, _ = net64.get_logits_values_and_hx(obs.double().cpu(), hx0.double().cpu(), prev_dones.cpu())
                lp = torch.log_softmax(logits, -1).gather(-1, actions.cpu().unsqueeze(-1)).squeeze(-1)
        assert float((v - values.cpu().double()).abs().max()) <= 1e-5
        assert float((lp - log_probs.cpu().double()).abs().max()) <= 1e-5
        assert bool(torch.isfinite(next_values).all())


@gpu
def test_lstm_host_env_rollout_learn_from_records_and_predict():
    """Host SyncVectorEnv CartPole: train() runs the fused forward per step with the packed state; learn() takes the reference's list
    of step records; predict() takes and returns hx [1, n, 2Hg] (None: zeros), h | c."""
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    from diamond.recurrent import RecurrentLSTMActorCriticNetwork
    N_, T, Hg = 8, 16, 24
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=2, total_steps=N_ * T * 2, gru_hidden_dim=Hg)
    agent = RecurrentPPO(lambda: envs.make("CartPole-v1"), cfg, network_cls=RecurrentLSTMActorCriticNetwork)
    before = {k: v.detach().clone() for k, v in agent.network.state_dict().items()}
    agent.train()
    assert torch.isfinite(agent.last_losses).all() and agent.current_hx.shape == (1, N_, 2 * Hg)
    _start(agent)
    ro = agent.rollout()
    records = list(ro)
    assert len(records) == T and records[0][9].shape == (1, N_, 2 * Hg)
    agent.learn(records)
    torch.cuda.synchronize()
    after = agent.network.state_dict()
    assert any(not torch.equal(before[k], after[k]) for k in before)
    assert all(torch.isfinite(v).all() for v in after.values()) and torch.isfinite(agent.last_losses).all()
    obs = np.random.default_rng(0).standard_normal((5, 4)).astype(np.float32)
    actions, hx = agent.predict(obs)
    assert actions.shape == (5,) and hx.shape == (1, 5, 2 * Hg) and isinstance(hx, np.ndarray)
    actions2, hx2 = agent.predict(obs, hx, np.array([True, False, False, False, False]))
    with torch.inference_mode():
        net = agent.network
        logits, _, ref = net.get_logits_values_and_hx(torch.as_tensor(obs, device=agent.device)[None], torch.as_tensor(hx, device=agent.device),
                                                      torch.tensor([[True, False, False, False, False]], device=agent.device))
    assert float(np.abs(hx2 - ref.cpu().numpy()).max()) <= 1e-5
    a_dev, h_dev = agent.predict(torch.as_tensor(obs, device=agent.device), torch.as_tensor(hx, device=agent.device))
    assert torch.is_tensor(a_dev) and h_dev.shape == (1, 5, 2 * Hg)


def _host_loop(agent, env_fn, num_envs, num_episodes, seed):
    from evaluate_oracle import EvalBook, quotas
    envs = env_fn(num_envs)
    book = EvalBook(quotas(num_episodes, num_envs))
    obs, _ = envs.reset(seed=seed)
    hx, prev = None, np.zeros(num_envs, dtype=bool)
    while book.remaining > 0:
        actions, hx = agent.predict(obs, hx, prev)
        nobs, rew, term, trunc, info = envs.step(actions)
        book.step(info.get("raw_rewards", rew), term, trunc)
        dones = term | trunc
        obs = envs.reset(options={"reset_mask": dones})[0] if dones.any() else nobs
        prev = dones
    return book.out_returns, book.out_lengths


@gpu
@pytest.mark.parametrize("kind,env_id", [("disc", "CartPole-v1"), ("cont", "Pendulum-v1")])
def test_lstm_evaluate_on_device_equals_host_loop(kind, env_id):
    agent, env_fn = _lstm_agent(kind, env_id)
    _start(agent)
    for _ in range(2):
        agent.learn(agent.rollout())
    res = agent.evaluate(10, num_envs=4, seed=77)
    ret, length = _host_loop(agent, env_fn, 4, 10, 77)
    assert np.array_equal(res["returns"], ret) and np.array_equal(res["lengths"], length)


@gpu
def test_lstm_evaluate_leaves_training_bit_identical():
    """k x (rollout + learn), evaluate(), k more == 2k x (rollout + learn): parameters, Adam state, environments, the packed state."""
    k = 2

    def run(with_eval):
        agent, _ = _lstm_agent("disc", "CartPole-v1", seed=13)
        _start(agent)
        for _ in range(k):
            agent.learn(agent.rollout())
        if with_eval:
            agent.evaluate(10, num_envs=5, seed=99)
            agent.evaluate(4, num_envs=4, deterministic=False)
        for _ in range(k):
            agent.learn(agent.rollout())
        torch.cuda.synchronize()
        eng = agent.engine
        return dict(P=eng.P.clone(), M=eng.M.clone(), V=eng.V.clone(), step=eng.adam_step, draws=eng.draws, hx=agent.current_hx.clone(),
                    envs={n: getattr(agent.envs, n).clone() for n in agent.envs.state_tensors})

    a, b = run(True), run(False)
    for key in ("P", "M", "V", "hx"):
        assert torch.equal(a[key], b[key]), key
    assert a["step"] == b["step"] and a["draws"] == b["draws"]
    for n in a["envs"]:
        assert torch.equal(a["envs"][n], b["envs"][n]), n


@gpu
def test_lstm_state_dict_loads_into_fresh_module_and_torch_lstm():
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork
    agent, _ = _lstm_agent("cont", "Pendulum-v1", seed=1, T=8)
    _start(agent)
    agent.learn(agent.rollout())
    sd = {k: v.detach().cpu().clone() for k, v in agent.network.state_dict().items()}
    fresh = RecurrentContinuousLSTMActorCriticNetwork(agent.envs.single_observation_space, agent.envs.single_action_space, agent.cfg)
    fresh.load_state_dict(sd)
    obs = torch.randn(5, 16, 3)
    with torch.inference_mode():
        a = agent.network.cpu().get_means_log_stds_values_and_hx(obs, None, None)
        b = fresh.get_means_log_stds_values_and_hx(obs, None, None)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    lstm = torch.nn.LSTM(agent.cfg.network_hidden_dim, agent.cfg.gru_hidden_dim)
    lstm.load_state_dict({k[len("lstm."):]: v for k, v in sd.items() if k.startswith("lstm.")})
    x = torch.randn(6, 4, agent.cfg.network_hidden_dim)
    with torch.no_grad():
        out, (h, c) = lstm(x)
        ours, hx = fresh.lstm(x, None, None)
    assert float((out - ours).abs().max()) <= 1e-6 and float((torch.cat([h, c], -1) - hx).abs().max()) <= 1e-6


@gpu
def test_custom_lstm_network_with_recurrent_state_dim_trains_on_autograd_engine():
    """A user's own LSTM network_cls (nn.LSTM inside, (h, c) packed into one tensor) declares recurrent_state_dim and trains on the
    autograd engine through the host rollout loop, learn() and predict()."""
    from diamond import RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.recurrent import RecurrentEngine

    class MyLSTMNet(torch.nn.Module):
        def __init__(self, observation_space, action_space, cfg):
            super().__init__()
            self.hg = 20
            self.recurrent_state_dim = 2 * self.hg
            self.base = torch.nn.Linear(int(np.prod(observation_space.shape)), 32)
            self.cell = torch.nn.LSTMCell(32, self.hg)
            self.actor_out_layer = torch.nn.Linear(self.hg, int(action_space.n))
            self.critic = torch.nn.Linear(self.hg, 1)

        def _core(self, obs, hx, dones):
            T, B = obs.shape[:2]
            s = torch.zeros(B, 2 * self.hg, device=obs.device) if hx is None else hx.reshape(B, 2 * self.hg)
            h, c = s[:, :self.hg], s[:, self.hg:]
            outs = []
            for t in range(T):
                if dones is not None:
                    keep = (~dones[t].to(torch.bool)).float().unsqueeze(-1)
                    h, c = h * keep, c * keep
                h, c = self.cell(torch.tanh(self.base(obs[t])), (h, c))
                outs.append(h)
            return torch.stack(outs), torch.cat([h, c], -1).unsqueeze(0)

        def get_values(self, obs, hx, dones):
            x, _ = self._core(obs, hx, dones)
            return self.critic(x).squeeze(-1)

        def get_logits_values_and_hx(self, obs, hx, dones):
            x, hx = self._core(obs, hx, dones)
            return self.actor_out_layer(x), self.critic(x).squeeze(-1), hx

    N_, T = 8, 8
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=5, total_steps=N_ * T * 3)
    agent = RecurrentPPO(DeviceVectorEnv.factory("CartPole-v1", seed=5), cfg, network_cls=MyLSTMNet)
    assert isinstance(agent.engine, RecurrentEngine) and agent.state_dim == 40
    before = {k: v.detach().clone() for k, v in agent.network.state_dict().items()}
    agent.train()
    torch.cuda.synchronize()
    assert agent.current_hx.shape == (1, N_, 40) and torch.isfinite(agent.last_losses).all()
    assert any(not torch.equal(before[k], v) for k, v in agent.network.state_dict().items())
    actions, hx = agent.predict(np.zeros((3, 4), np.float32))
    assert hx.shape == (1, 3, 40)


# ---------------------------------------------------------------- learning ---------------------------------------------------------
# Budgets and bounds from 5-seed runs of tests/lstm_learning_curve.py on one B200 at a 1000 W power limit (DESIGN.md §8d): CartPole,
# 150 rollouts, last-20-episode means 388 / 500 / 29 / 387 / 213 for seeds 0-4 (seed 2 has not learned yet; the test runs seed 0);
# normalised Pendulum, 400 rollouts, -400 / -247 / -277 / -260 / -158 (random policies return about -1230).
CARTPOLE_ROLLOUTS, CARTPOLE_BOUND = 150, 100.0
PENDULUM_ROLLOUTS, PENDULUM_BOUND = 400, -700.0


@gpu
def test_lstm_recurrent_agent_learns_device_cartpole():
    from diamond import RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.recurrent import RecurrentLSTMActorCriticNetwork
    N_, T = 64, 32
    cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, num_minibatches=4, verbose=False, seed=0,
                             total_steps=N_ * T * CARTPOLE_ROLLOUTS)
    agent = RecurrentPPO(DeviceVectorEnv.factory("CartPole-v1", seed=0), cfg, network_cls=RecurrentLSTMActorCriticNetwork)
    agent.train()
    returns = agent.ticker.logs["episode_returns"]
    assert len(returns) >= 20
    assert np.mean(returns[-20:]) > CARTPOLE_BOUND, np.mean(returns[-20:])


@gpu
def test_lstm_gaussian_agent_learns_normalised_device_pendulum():
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork
    N_, T = 64, 32
    cfg = RecurrentContinuousPPOConfig(num_envs=N_, rollout_steps=T, num_minibatches=4, verbose=False, seed=0,
                                       total_steps=N_ * T * PENDULUM_ROLLOUTS)
    env_fn = DeviceVectorEnv.factory("Pendulum-v1", seed=0, normalize_observation=True, normalize_reward=True)
    agent = RecurrentContinuousPPO(env_fn, cfg, network_cls=RecurrentContinuousLSTMActorCriticNetwork)
    agent.train()
    returns = agent.ticker.logs["episode_returns"]
    assert len(returns) >= 20
    assert np.mean(returns[-20:]) > PENDULUM_BOUND, np.mean(returns[-20:])


@gpu
def test_dp_two_gpus_recurrent_lstm():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tests", "dp_equivalence_lstm.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "OK" in r.stdout and "FAIL" not in r.stdout
