"""RecurrentContinuousPPO: the Gaussian-policy recurrent network (dppo_rnn_desc.continuous = 1) through the C ABI against a float64
CPU autograd reference on every GRU scan branch and both head kernels, and the agent on device and host environments.

The reference is diamond.recurrent.RecurrentContinuousActorCriticNetwork in float64 on the CPU, loaded from the same flat fp32
buffer, with the Gaussian PPO loss of continuous_ppo.py written out as in oracle/ppo_oracle.py loss_and_grads.  The scan-branch
and cluster-plan mirrors, the inputs' conventions and the bars are those of test_rnn_kernels_gpu.py / test_rnn_wide_gpu.py."""
import math
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_rnn_kernels_gpu import CLIP, BETA, VW, GRAD_TOL, cuda, make_hyper, nerr, scan_branch, envs_per_block, ALL_BRANCHES
from test_rnn_wide_gpu import branch as cluster_branch

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def head_kernel(H, A):
    """heads.cu launch_head_train_kernel: the role-split kernel at H = 128 / 256 with A <= 4 (rows 16-byte aligned, always so
    here), the generic one otherwise."""
    return "split" if H in (128, 256) and A <= 4 else "generic"


def case_branch(N, Hg):
    return scan_branch(N, Hg) if Hg <= 128 else cluster_branch(N, Hg)


# One row per case: the scan branch it is meant to run (single-CTA kernels as in test_rnn_kernels_gpu.py, cluster kernels as in
# test_rnn_wide_gpu.py), then the shapes.  opts: "hx0" non-zero initial state, "dones" resets, "norm" advantage normalisation from
# fp64 statistics, "den2" loss denominator 2 M.
CASES = [
    # id        branch    D    H   Hg   A   T     N   opts
    ("hg1",     "smem",   3,  32,   1,  1, 33,  257, "hx0 dones"),
    ("hg8",     "warp8",  5, 128,   8,  3, 64,   17, "hx0 dones"),
    ("hg10",    "smem",   3, 200,  10,  5,  2,   26, "dones den2"),
    ("hg12",    "tiled1", 6,  64,  12, 32, 33,   22, "hx0 dones"),
    ("hg16",    "warp16", 3,  64,  16,  1, 64,    9, "hx0 dones norm"),
    ("hg32",    "warp32", 8,  32,  32,  4, 33,    5, "hx0 dones den2"),
    ("hg50",    "smem",   6, 200,  50,  2, 33,    6, "hx0 dones norm"),
    ("hg64-e2", "tiled2", 8,  64,  64,  4,  3, 1801, "hx0 dones norm"),
    ("hg64-e4", "tiled4", 8, 256,  64,  2,  4, 4099, "hx0 dones"),
    ("hg128",   "tiled1", 4, 160, 128, 32,  2,    3, "hx0 dones den2"),
    ("hg256",   "c8e1",   6, 128, 256,  2, 64,    5, "hx0 dones"),
    ("hg512",   "c16e1",  5, 256, 512,  3,  1,   19, "hx0 dones norm"),
    ("null",    "warp16", 4,  32,  16,  2,  5,   40, ""),
]
CASE_IDS = [c[0] for c in CASES]


# ---------------------------------------------------------------- CPU: layout, module, case table ----------------------------
def test_continuous_layout_matches_module():
    """The continuous layout has the module's 15 tensors (6 499 parameters at D = 3, H = 64, Hg = 16, A = 1) at distinct,
    non-overlapping offsets that are multiples of 4, and state_dict keys equal the module's."""
    from diamond import _native as Nt
    from diamond.config import RecurrentContinuousPPOConfig
    from diamond.recurrent import RecurrentContinuousActorCriticNetwork, rnn_param_slices
    for D, H, Hg, A in ((3, 64, 16, 1), (5, 200, 50, 32), (8, 128, 256, 4)):
        desc = Nt.RnnDesc(D, H, Hg, A, 1)
        lay = Nt.rnn_layout(desc)
        sl = rnn_param_slices(desc, lay)
        net = RecurrentContinuousActorCriticNetwork(SimpleNamespace(shape=(D,)), SimpleNamespace(shape=(A,)),
                                                    RecurrentContinuousPPOConfig(network_hidden_dim=H, gru_hidden_dim=Hg))
        params = dict(net.named_parameters())
        assert len(sl) == 15 and set(sl) == set(params) == set(net.state_dict())
        assert all(tuple(params[k].shape) == shape for k, (_, shape) in sl.items())
        spans = sorted((off, off + int(np.prod(shape))) for off, shape in sl.values())
        assert all(off % 4 == 0 for off, _ in spans)
        assert all(a_end <= b_off for (_, a_end), (b_off, _) in zip(spans, spans[1:]))
        assert spans[-1][1] <= lay.total and lay.log_std == sl["actor_log_std"][0] and lay.log_std > lay.bc
        if (D, H, Hg, A) == (3, 64, 16, 1):
            assert sum(p.numel() for p in params.values()) == 6499


def test_discrete_layout_unchanged():
    """continuous = 0 (what existing callers leave in the new field): every offset and the total are today's, log_std is -1."""
    from diamond import _native as Nt
    for D, H, Hg, A in ((4, 64, 16, 2), (3, 200, 50, 7), (8, 128, 512, 32)):
        up = lambda n: (n + 3) // 4 * 4
        names = ["w1", "b1", "wih", "whh", "bih", "bhh", "w3", "b3", "wa", "ba", "wc", "bc"]
        sizes = [H * D, H, 3 * Hg * H, 3 * Hg * Hg, 3 * Hg, 3 * Hg, 2 * H * Hg, 2 * H, A * H, A, H, 1]
        lay = Nt.rnn_layout(Nt.RnnDesc(D, H, Hg, A))
        o = 0
        for n, sz in zip(names, sizes):
            assert getattr(lay, n) == o, n
            o += up(sz)
        assert lay.total == o and lay.log_std == -1


def test_case_table_covers_branches_and_head_kernels():
    """CPU: each case runs the scan branch it names; together they run all seven single-CTA scan pairs and both cluster widths,
    the role-split head kernel at H = 128 and 256 and the generic one (H = 200 among them), A = 1 and A = 32."""
    seen = set()
    for cid, br, D, H, Hg, A, T, N, opts in CASES:
        assert case_branch(N, Hg) == br, cid
        seen.add(br)
    assert ALL_BRANCHES <= seen and {"c8e1", "c16e1"} <= seen
    assert {c[4] for c in CASES} >= {256, 512}
    heads = {(head_kernel(c[3], c[5]), c[3]) for c in CASES}
    assert {("split", 128), ("split", 256), ("generic", 200)} <= heads
    assert {1, 32} <= {c[5] for c in CASES}
    one_past = {c[1] for c in CASES if c[4] <= 128 and c[7] % envs_per_block(c[7], c[4]) == 1}
    assert {"warp8", "warp32", "smem"} <= one_past
    opts = " ".join(c[8] for c in CASES).split()
    assert {"hx0", "dones", "norm", "den2"} <= set(opts) and any(c[8] == "" for c in CASES)


def test_discrete_network_still_refuses_box_actions():
    """RecurrentActorCriticNetwork (RecurrentPPO's default) keeps its assertion on a Box action space."""
    from diamond.config import RecurrentPPOConfig
    from diamond.recurrent import RecurrentActorCriticNetwork
    with pytest.raises(AssertionError, match="Only Discrete action spaces are supported."):
        RecurrentActorCriticNetwork(SimpleNamespace(shape=(3,)), SimpleNamespace(shape=(1,)), RecurrentPPOConfig())


# ---------------------------------------------------------------- inputs and the float64 reference -----------------------------
def make_inputs(case, seed=0):
    cid, br, D, H, Hg, A, T, N, opts = case
    rng = np.random.default_rng(1000 * CASE_IDS.index(cid) + seed + 555)
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    desc = Nt.RnnDesc(D, H, Hg, A, 1)
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
    hx0 = (0.5 * rng.standard_normal((N, Hg))).astype(np.float32) if "hx0" in opts else None
    dones = None
    if "dones" in opts:
        dones = rng.random((T, N)) < 0.15
        dones[np.arange(T), rng.integers(0, N, T)] = True
        dones[0, : max(1, N // 3)] = True
    adv = rng.standard_normal((T, N)).astype(np.float32)
    ret = rng.standard_normal((T, N)).astype(np.float32)
    return SimpleNamespace(case=case, desc=desc, lay=lay, slices=slices, flat=flat, obs=obs, hx0=hx0, dones=dones, adv=adv, ret=ret,
                           rng=rng, D=D, H=H, Hg=Hg, A=A, T=T, N=N)


def reference_network(x):
    from diamond.config import RecurrentContinuousPPOConfig
    from diamond.recurrent import RecurrentContinuousActorCriticNetwork
    cfg = RecurrentContinuousPPOConfig(network_hidden_dim=x.H, gru_hidden_dim=x.Hg)
    net = RecurrentContinuousActorCriticNetwork(SimpleNamespace(shape=(x.D,)), SimpleNamespace(shape=(x.A,)), cfg).double()
    params = dict(net.named_parameters())
    with torch.no_grad():
        for name, (off, shape) in x.slices.items():
            params[name].copy_(torch.as_tensor(x.flat[off:off + int(np.prod(shape))].astype(np.float64)).reshape(shape))
    return net


def reference_forward(x, net, with_state=True):
    obs = torch.as_tensor(x.obs, dtype=torch.float64)
    hx = torch.as_tensor(x.hx0, dtype=torch.float64).unsqueeze(0) if (with_state and x.hx0 is not None) else None
    dn = torch.as_tensor(x.dones) if (with_state and x.dones is not None) else None
    return net.get_means_log_stds_values_and_hx(obs, hx, dn)


def normal_log_prob(mean, log_std, actions):
    return (-((actions - mean) ** 2) / (2 * torch.exp(2 * log_std)) - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)


def set_actions_and_old_log_probs(x, mean, log_std):
    """actions drawn from the fp64 policy; old log-probs placed so that every ratio sits at least 1e-2 from the clip edges (as
    test_rnn_kernels_gpu.set_old_log_probs does)."""
    B, A = x.T * x.N, x.A
    m, ls = mean.detach().reshape(B, A), log_std.detach().reshape(B, A)
    x.actions = (m + ls.exp() * torch.as_tensor(x.rng.standard_normal((B, A)))).numpy().astype(np.float32)
    new_lp = normal_log_prob(m, ls, torch.as_tensor(x.actions.astype(np.float64))).numpy()
    u = x.rng.random(B)
    ratio = np.where(u < 0.5, x.rng.uniform(1 - CLIP + 0.01, 1 + CLIP - 0.01, B),
                     np.where(u < 0.75, x.rng.uniform(0.5, 1 - CLIP - 0.01, B), x.rng.uniform(1 + CLIP + 0.01, 1.6, B)))
    x.old_lp = (new_lp - np.log(ratio)).astype(np.float32)
    lr = new_lp - x.old_lp.astype(np.float64)
    edge = np.minimum(np.abs(np.exp(lr) - (1 - CLIP)), np.abs(np.exp(lr) - (1 + CLIP)))
    assert edge.min() >= 1e-3


def reference_loss(x, mean, log_std, values, rows, adv_norm, den):
    """Gaussian PPO loss (continuous_ppo.py; oracle/ppo_oracle.py loss_and_grads) on rows `rows` of the flattened outputs, float64."""
    B, A = x.T * x.N, x.A
    m, ls = mean.reshape(B, A)[rows], log_std.reshape(B, A)[rows]
    v = values.reshape(B)[rows]
    act = torch.as_tensor(x.actions.reshape(B, A)[rows].astype(np.float64))
    old = torch.as_tensor(x.old_lp[rows].astype(np.float64))
    a = torch.as_tensor(x.adv.reshape(B).astype(np.float64))
    if adv_norm:
        mu = a.mean()
        a = (a - mu) / (torch.sqrt(((a - mu) ** 2).sum() / (B - 1)) + 1e-6)
    a = a[rows]
    ret = torch.as_tensor(x.ret.reshape(B)[rows].astype(np.float64))
    ratio = torch.exp(normal_log_prob(m, ls, act) - old)
    pol = torch.max(-a * ratio, -a * torch.clamp(ratio, 1 - CLIP, 1 + CLIP)).sum() / den
    val = 0.5 * ((v - ret) ** 2).sum() / den
    ent = (0.5 + 0.5 * math.log(2 * math.pi) + ls).sum(-1).sum() / den
    total = pol + VW * val - BETA * ent
    return total, [pol, val, ent, total]


@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as Nt
    return Nt.get_context(0)


def to_device(x):
    B = x.T * x.N
    a64 = x.adv.astype(np.float64).reshape(-1)
    return SimpleNamespace(P=cuda(x.flat), obs=cuda(x.obs), pd=cuda(x.dones, torch.uint8), hx0=cuda(x.hx0),
                           actions=cuda(x.actions.reshape(B, x.A)), old_lp=cuda(x.old_lp), adv=cuda(x.adv.reshape(B)),
                           ret=cuda(x.ret.reshape(B)), stats=cuda(np.array([a64.sum(), (a64 ** 2).sum()]), torch.float64))


def check_grad_vs_fp64(ctx, case):
    cid, br, D, H, Hg, A, T, N, opts = case
    x = make_inputs(case)
    B = T * N
    net = reference_network(x)
    mean, log_std, values, _ = reference_forward(x, net)
    set_actions_and_old_log_probs(x, mean, log_std)
    d = to_device(x)
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
        total, ref_losses = reference_loss(x, mean, log_std, values, rsel, adv_norm, den)
        total.backward(retain_graph=True)
        ref = {n: p.grad.numpy() for n, p in net.named_parameters()}
        hyper = make_hyper(M, den, adv_norm, B)
        hyper.grad_sumsq = sumsq.data_ptr()
        ws = torch.empty(ctx.rnn_workspace_bytes(x.desc, T, N, M, True) // 4 + 64, device="cuda")
        grads = torch.full((int(x.lay.total),), 7.0, device="cuda")
        losses = torch.zeros(4, device="cuda")
        ctx.rnn_grad_minibatch(x.desc, d.P, grads, d.obs, d.pd, d.hx0, T, N, d.actions, d.old_lp, d.adv, d.ret, d.stats,
                               cuda(rows, torch.int32), M, hyper, losses, ws)
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
        ctx.clip_adam_step(d.P.clone(), grads.clone(), z, z.clone(), hyper, adam_ws, gn)
        torch.cuda.synchronize()
        assert abs(float(gn) - ref_norm) <= GRAD_TOL * ref_norm, (where, float(gn), ref_norm)


# ---------------------------------------------------------------- GPU: kernels against float64 --------------------------------
@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_gaussian_rnn_grad_minibatch_vs_fp64(ctx, case):
    """dppo_rnn_grad_minibatch with continuous = 1, whole rollout (idx NULL) and a permutation slice: all 15 gradient tensors
    including actor_log_std (2e-5 of each tensor's largest entry), the losses (rtol 1e-5), zero padding and the clip norm."""
    check_grad_vs_fp64(ctx, case)


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_gaussian_rnn_forward_vs_fp64(ctx, case):
    """dppo_rnn_forward with continuous = 1, heads 1, 2 and 3, with and without resets / initial state: means, values and the final
    hidden state within 1e-5 of float64."""
    cid, br, D, H, Hg, A, T, N, opts = case
    x = make_inputs(case, seed=1)
    net = reference_network(x)
    ws = torch.empty(ctx.rnn_workspace_bytes(x.desc, T, N, T * N, False) // 4 + 64, device="cuda")
    P, obs = cuda(x.flat), cuda(x.obs)
    tol = lambda ref: 1e-5 * max(1.0, float(np.abs(ref).max()))
    for with_state in (True, False):
        with torch.no_grad():
            rm, _, rv, rh = (t.numpy() for t in reference_forward(x, net, with_state))
        pd = cuda(x.dones, torch.uint8) if with_state else None
        hx0 = cuda(x.hx0) if with_state else None
        for heads in (1, 2, 3):
            means = torch.full((T, N, A), float("nan"), device="cuda") if heads & 1 else None
            values = torch.full((T, N), float("nan"), device="cuda") if heads & 2 else None
            hx = torch.full((N, Hg), float("nan"), device="cuda")
            ctx.rnn_forward(x.desc, P, obs, pd, hx0, T, N, heads, means, values, hx, ws)
            torch.cuda.synchronize()
            where = (cid, with_state, heads)
            if heads & 1:
                assert np.abs(means.cpu().numpy() - rm).max() <= tol(rm), where
            if heads & 2:
                assert np.abs(values.cpu().numpy() - rv).max() <= tol(rv), where
            assert np.abs(hx.cpu().numpy() - rh[0]).max() <= tol(rh), where


@gpu
@pytest.mark.parametrize("D,H,Hg,A,bound", [(4, 64, 16, 33, "32"), (4, 513, 16, 2, "512"), (4, 64, 513, 2, "512"),
                                            (4, 512, 16, 11, "200 KB")])
def test_gaussian_rnn_refusals(ctx, D, H, Hg, A, bound):
    """A > 32, H > 512, Hg > 512 and a head-kernel accumulator band beyond 200 KB are refused with a NativeError naming the bound,
    before anything is launched; the same context then computes a correct gradient."""
    from diamond import _native as Nt
    desc = Nt.RnnDesc(D, H, Hg, A, 1)
    lay = Nt.rnn_layout(desc)
    T, N = 2, 3
    B = T * N
    P = torch.zeros(int(lay.total), device="cuda")
    ws = torch.empty(ctx.rnn_workspace_bytes(desc, T, N, B, True) // 4 + 64, device="cuda")
    launches = ctx.launches
    obs = torch.zeros(T, N, D, device="cuda")
    if bound != "200 KB":
        with pytest.raises(Nt.NativeError, match=bound):
            ctx.rnn_forward(desc, P, obs, None, None, T, N, 3, torch.empty(T, N, A, device="cuda"), torch.empty(T, N, device="cuda"),
                            torch.empty(N, Hg, device="cuda"), ws)
    hyper = make_hyper(B, B, False, B)
    f = lambda *s: torch.zeros(*s, device="cuda")
    with pytest.raises(Nt.NativeError, match=bound):
        ctx.rnn_grad_minibatch(desc, P, f(int(lay.total)), obs, None, None, T, N, f(B, A), f(B), f(B), f(B), None, None, B, hyper,
                               f(4), ws)
    assert ctx.launches == launches
    check_grad_vs_fp64(ctx, CASES[CASE_IDS.index("hg16")])


# ---------------------------------------------------------------- GPU: agent level ---------------------------------------------
def _synthetic_rollout(T, N_, D, A, Hg, dev, seed):
    from diamond.recurrent import RecurrentRollout
    gen = torch.Generator(device=dev).manual_seed(seed)
    ro = RecurrentRollout(T, N_, D, Hg, dev, A)
    ro.obs.normal_(generator=gen); ro.actions.normal_(generator=gen); ro.rewards.normal_(generator=gen)
    ro.terminations.copy_((torch.rand(T, N_, device=dev, generator=gen) < 0.1).float()); ro.truncations.zero_()
    ro.prev_dones.copy_(torch.rand(T, N_, device=dev, generator=gen) < 0.1)
    ro.log_probs.copy_(-0.5 * (ro.actions ** 2).sum(-1) - 0.5 * A * math.log(2 * math.pi))
    ro.values.normal_(generator=gen); ro.next_values.normal_(generator=gen)
    ro.hx0.normal_(generator=gen); ro.filled = T
    return ro


@gpu
@pytest.mark.parametrize("Hg,N_,T", [(16, 24, 16), (64, 20, 9), (256, 38, 19)])
def test_gaussian_fused_engine_matches_autograd_engine(Hg, N_, T):
    """RecurrentContinuousPPO's fused engine (default network) equals the same network under torch autograd (RecurrentEngine, a
    subclass of the default network) on the same rollout: one learn() of 2 epochs x 2 minibatches, parameters and losses within 1e-4,
    at the warp (16), tiled (64) and cluster (256) GRU widths."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig, envs
    from diamond.recurrent import RecurrentContinuousActorCriticNetwork, FusedRecurrentEngine, RecurrentEngine

    class Same(RecurrentContinuousActorCriticNetwork):
        pass

    D, A, H = 6, 3, 64
    agents = []
    for cls in (RecurrentContinuousActorCriticNetwork, Same):
        cfg = RecurrentContinuousPPOConfig(num_envs=N_, rollout_steps=T, num_epochs=2, num_minibatches=2, verbose=False,
                                           network_hidden_dim=H, gru_hidden_dim=Hg, seed=4, total_steps=N_ * T * 100)
        agents.append(RecurrentContinuousPPO(lambda: envs.SyntheticEnv(D, A, continuous=True), cfg, network_cls=cls))
    fused, auto = agents
    assert isinstance(fused.engine, FusedRecurrentEngine) and isinstance(auto.engine, RecurrentEngine)
    with torch.no_grad():
        fused.network.actor_log_std.copy_(torch.tensor([[-0.3, 0.1, -0.6]]))
    auto.network.load_state_dict(fused.network.state_dict())
    ro = _synthetic_rollout(T, N_, D, A, Hg, fused.device, Hg)
    for ag in (fused, auto):
        np.random.seed(8)
        ag.learn(ro)
    torch.cuda.synchronize()
    for (k, p), (_, q) in zip(fused.network.named_parameters(), auto.network.named_parameters()):
        err = float((p - q).abs().max() / q.abs().max().clamp_min(1e-12))
        assert err <= 1e-4, (k, err)
    assert float((fused.last_losses - auto.last_losses).abs().max()) <= 1e-4


@gpu
def test_gaussian_device_rollout_graph_replay_and_module():
    """Device Pendulum-v1 rollout (odd T, so the hidden state ping-pongs): the CUDA-graph replay (from the third rollout) records
    exactly what eager launches record, and the recorded values and Normal(mean, exp(log_std)).log_prob(a).sum(-1) are what the
    float64 module computes from the recorded sequence, to 1e-5."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    N_, T, Hg = 48, 17, 16
    recs = []
    for use_graphs in (True, False):
        cfg = RecurrentContinuousPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=6, total_steps=N_ * T * 100,
                                           gru_hidden_dim=Hg)
        agent = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=6), cfg)
        with torch.no_grad():
            agent.network.actor_log_std.fill_(-0.4)
        agent.engine.use_graphs = use_graphs
        agent.ticker = None
        agent.current_observations, _ = agent.envs.reset(seed=6)
        agent.prev_dones = np.zeros(N_, dtype=bool)
        agent.current_hx = torch.zeros(1, N_, Hg, device=agent.device)
        out = []
        for _ in range(5):
            ro = agent.rollout()
            out.append([getattr(ro, k).clone() for k in ("obs", "actions", "rewards", "terminations", "truncations", "prev_dones",
                                                         "log_probs", "values", "next_values", "hx0")])
        torch.cuda.synchronize()
        if use_graphs:
            assert agent._ro_graph is not None, "graph path was not taken"
            net64 = agent.network.double().cpu()
        recs.append(out)
    for a, b in zip(*recs):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    assert out[0][1].shape == (T, N_, 1) and out[0][1].dtype == torch.float32
    for obs, actions, rew, term, trunc, prev_dones, log_probs, values, next_values, hx0 in recs[0]:
        with torch.inference_mode():
            mean, ls, v, _ = net64.get_means_log_stds_values_and_hx(obs.double().cpu(), hx0.double().cpu(), prev_dones.cpu())
        lp = torch.distributions.Normal(mean, ls.exp()).log_prob(actions.double().cpu()).sum(-1)
        assert float((v - values.cpu().double()).abs().max()) <= 1e-5
        assert float((lp - log_probs.cpu().double()).abs().max()) <= 1e-5
        assert bool(torch.isfinite(next_values).all())


@gpu
def test_gaussian_host_env_rollout_and_learn_from_records():
    """Host SyncVectorEnv (envs.make("Pendulum-v1")): train() runs the fused forward + dppo_sample_gaussian per step; learn() also
    takes the rollout as the reference's list of step records.  Parameters move and stay finite, losses are finite."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig, envs
    N_, T = 8, 16
    cfg = RecurrentContinuousPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=2, total_steps=N_ * T * 2)
    agent = RecurrentContinuousPPO(lambda: envs.make("Pendulum-v1"), cfg)
    before = {k: v.detach().clone() for k, v in agent.network.state_dict().items()}
    agent.train()
    assert torch.isfinite(agent.last_losses).all()
    agent.current_observations, _ = agent.envs.reset(seed=3)
    agent.prev_dones = np.zeros(N_, dtype=bool)
    agent.current_hx = torch.zeros(1, N_, cfg.gru_hidden_dim, device=agent.device)
    ro = agent.rollout()
    records = list(ro)
    assert len(records) == T and records[0][1].shape == (N_, 1)
    agent.learn(records)
    torch.cuda.synchronize()
    after = agent.network.state_dict()
    assert any(not torch.equal(before[k], after[k]) for k in before)
    assert all(torch.isfinite(v).all() for v in after.values()) and torch.isfinite(agent.last_losses).all()


@gpu
def test_recurrent_ppo_refuses_box_action_space():
    from diamond import RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    with pytest.raises(AssertionError, match="Only Discrete action spaces are supported."):
        RecurrentPPO(DeviceVectorEnv.factory("Pendulum-v1"), RecurrentPPOConfig(verbose=False))


@gpu
def test_gaussian_checkpoint_state_dict_loads_into_fresh_module():
    """The agent's state_dict (views of the flat buffer) loads into a plain torch module, which then computes the same outputs."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.recurrent import RecurrentContinuousActorCriticNetwork
    cfg = RecurrentContinuousPPOConfig(num_envs=16, rollout_steps=8, verbose=False, seed=1, total_steps=16 * 8 * 2)
    agent = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=1), cfg)
    agent.train()
    sd = {k: v.detach().cpu().clone() for k, v in agent.network.state_dict().items()}
    fresh = RecurrentContinuousActorCriticNetwork(agent.envs.single_observation_space, agent.envs.single_action_space, cfg)
    fresh.load_state_dict(sd)
    obs = torch.randn(5, 16, 3)
    with torch.inference_mode():
        a = agent.network.cpu().get_means_log_stds_values_and_hx(obs, None, None)
        b = fresh.get_means_log_stds_values_and_hx(obs, None, None)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# Budget and bound from the learning curve of tests/rnn_gaussian_learning_curve.py (one B200 at a 1000 W power limit, DESIGN.md §8):
# device Pendulum-v1, 64 environments x 32 steps, gamma 0.9, lr 1e-3, 4 minibatches.  Random policies return about -1230; over rollouts
# 181-200 seeds 0-4 returned -190 / -242 / -203 / -284 / -222 (about 1.1 s of training).  Later windows dip as low as -943, so the
# budget stops at 200 rollouts.
LEARN_ROLLOUTS = 200
LEARN_BOUND = -600.0


@gpu
def test_gaussian_recurrent_agent_learns_device_pendulum():
    """RecurrentContinuousPPO on device Pendulum-v1 improves the mean episode return past a bound a random policy does not reach."""
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    N_, T = 64, 32
    cfg = RecurrentContinuousPPOConfig(num_envs=N_, rollout_steps=T, num_minibatches=4, gamma=0.9, lr=1e-3, verbose=False, seed=0,
                                       total_steps=N_ * T * LEARN_ROLLOUTS)
    agent = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=0), cfg)
    agent.train()
    returns = agent.ticker.logs["episode_returns"]
    assert len(returns) >= 20
    assert np.mean(returns[-20:]) > LEARN_BOUND, np.mean(returns[-20:])


@gpu
def test_dp_two_gpus_recurrent_gaussian():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tests", "dp_equivalence_recurrent_gaussian.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "OK" in r.stdout and "FAIL" not in r.stdout
