"""GRU widths 129-512 (csrc/rnn.cu cluster scans: W_hh split by hidden unit over the CTAs of a thread-block cluster, the hidden state
exchanged over distributed shared memory) through the C ABI and RecurrentPPO, against float64 CPU references.

The float64 reference and the PPO loss are those of test_rnn_kernels_gpu.py.  The mirror below restates the launch plan of the
cluster scans (rnn.cu cluster_plan) so that the case table can name, and a CPU test can check, the cluster size C, the units per
CTA U, the environments per thread E and the environments per cluster each case runs."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_rnn_kernels_gpu import (cuda, device_grad, make_hyper, nerr, reference_forward, reference_loss, reference_network,
                                  set_old_log_probs, to_device)

gpu = pytest.mark.gpu


# ---------------------------------------------------------------- mirror of rnn.cu cluster_plan ------------------------------
SMEM_FLOATS = 227 * 1024 // 4                           # rnn.cu kScanSmemFloats
MAX_GROUPS = 8                                          # rnn.cu kClusterMaxGroups


def cluster_plan(N, Hg):
    """(C, U, E, G, clusters): CTAs per cluster, hidden units per CTA, environments per thread, thread groups per CTA, clusters."""
    assert 128 < Hg <= 512
    C = 8 if Hg <= 256 else 16
    U = -(-Hg // C)
    HP = (Hg + 3) & ~3
    fwd = lambda e: 3 * U * (HP + 4) + 2 * e * HP       # rnn.cu cluster_fwd_smem_floats
    bwd = lambda e: 3 * U * Hg + e * (3 * U + 2 * C * U)  # rnn.cu cluster_bwd_smem_floats
    cap = 1
    while fwd(cap + 1) <= SMEM_FLOATS and bwd(cap + 1) <= SMEM_FLOATS:
        cap += 1
    slots = 148 // C
    ec = min(-(-N // slots), cap, 4 * MAX_GROUPS)
    E = 1 if ec <= MAX_GROUPS else 2 if ec <= 2 * MAX_GROUPS else 4
    G = -(-ec // E)
    while G > 1 and G * E > cap:
        G -= 1
    return C, U, E, G, -(-N // (G * E))


def branch(N, Hg):
    C, U, E, G, _ = cluster_plan(N, Hg)
    return f"c{C}e{E}"


def envs_per_cluster(N, Hg):
    C, U, E, G, _ = cluster_plan(N, Hg)
    return G * E


# One row per case: the cluster branch (C CTAs per cluster, E environments per thread), then the shapes.  N is one environment
# past a cluster boundary where the plan allows it; H = 128 with A <= 4 takes the role-split head kernel, every other (H, A) the
# generic one.  opts as in test_rnn_kernels_gpu.py: "hx0", "dones", "norm" (advantage normalisation), "den2" (denominator 2 M).
CASES = [
    # id          branch   D    H   Hg  A   T    N   opts
    ("hg129",     "c8e1",  4, 128, 129, 3, 33,  19, "hx0 dones"),
    ("hg130",     "c8e1",  5,  64, 130, 5,  2,  19, "hx0 dones norm"),
    ("hg192-e2",  "c8e2",  3,  32, 192, 4,  3, 161, "hx0 dones den2"),
    ("hg256",     "c8e1",  6, 128, 256, 2, 64,   5, "hx0 dones"),
    ("hg256-e4",  "c8e4",  4,  64, 256, 3,  2, 577, "dones norm"),
    ("hg257",     "c16e1", 4,  64, 257, 6, 33,  19, "hx0 dones"),
    ("hg300-e2",  "c16e2", 3, 200, 300, 5,  2,  97, "hx0 dones den2"),
    ("hg512",     "c16e1", 5, 128, 512, 4,  1,  19, "hx0 dones norm"),
    ("hg512-t64", "c16e1", 4,  96, 512, 3, 64,   6, ""),
]
CASE_IDS = [c[0] for c in CASES]


def test_case_table_covers_cluster_shapes():
    """CPU: each case runs the branch it names; together they run C = 8 and 16 with E = 1, 2 and 4, Hg = 129 / 256 / 512, widths C
    does not divide that are not multiples of 4, a last cluster holding one environment, T = 1, 2, odd and 64, both head kernels
    and every option."""
    for cid, br, D, H, Hg, A, T, N, opts in CASES:
        assert branch(N, Hg) == br, (cid, cluster_plan(N, Hg))
        C, U, E, G, _ = cluster_plan(N, Hg)
        assert U <= 32 and G * U <= 256
    seen = {c[1] for c in CASES}
    assert {"c8e1", "c8e2", "c8e4", "c16e1", "c16e2"} <= seen
    hgs = {c[4] for c in CASES}
    assert {129, 256, 512} <= hgs
    for C in (8, 16):                                   # a width C does not divide, not a multiple of 4 (e.g. 130, 257)
        assert any(cluster_plan(N, Hg)[0] == C and Hg % C and Hg % 4 for _, _, D, H, Hg, A, T, N, _ in CASES), C
    assert any(N % envs_per_cluster(N, Hg) == 1 for _, _, D, H, Hg, A, T, N, _ in CASES if cluster_plan(N, Hg)[0] == 8)
    assert any(N % envs_per_cluster(N, Hg) == 1 for _, _, D, H, Hg, A, T, N, _ in CASES if cluster_plan(N, Hg)[0] == 16)
    Ts = {c[6] for c in CASES}
    assert {1, 2, 64} <= Ts and any(t % 2 == 1 and t > 16 for t in Ts)
    assert any(H == 128 and A <= 4 for _, _, D, H, Hg, A, T, N, _ in CASES)
    assert any(not (H == 128 and A <= 4) for _, _, D, H, Hg, A, T, N, _ in CASES)
    opts = " ".join(c[8] for c in CASES).split()
    assert {"hx0", "dones", "norm", "den2"} <= set(opts) and any(c[8] == "" for c in CASES)
    # the shapes of the latency script and the agent-level tests: defaults (N = 32) spread two environments per cluster; at
    # Hg = 512 shared memory holds 8 environments per 16-CTA cluster
    assert cluster_plan(32, 256)[2:] == (1, 2, 16) and cluster_plan(32, 512)[2:] == (1, 4, 8)
    assert cluster_plan(4096, 512)[2:] == (1, 8, 512) and cluster_plan(4096, 256)[2:4] == (4, 8)


# ---------------------------------------------------------------- inputs ------------------------------------------------------
def make_inputs(case, seed=0):
    cid, br, D, H, Hg, A, T, N, opts = case
    rng = np.random.default_rng(1000 * CASE_IDS.index(cid) + seed + 77)
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    desc = Nt.RnnDesc(D, H, Hg, A)
    lay = Nt.rnn_layout(desc)
    slices = rnn_param_slices(desc, lay)
    flat = np.zeros(int(lay.total), np.float32)
    for name, (off, shape) in slices.items():
        w = rng.standard_normal(shape) / np.sqrt(shape[1]) if len(shape) == 2 else 0.3 * rng.standard_normal(shape)
        flat[off:off + int(np.prod(shape))] = w.reshape(-1)
    obs = rng.standard_normal((T, N, D)).astype(np.float32)
    hx0 = (0.5 * rng.standard_normal((N, Hg))).astype(np.float32) if "hx0" in opts else None
    dones = None
    if "dones" in opts:
        dones = rng.random((T, N)) < 0.15
        dones[np.arange(T), rng.integers(0, N, T)] = True
        dones[0, : max(1, N // 3)] = True
    actions = rng.integers(0, A, (T, N)).astype(np.int32)
    adv = rng.standard_normal((T, N)).astype(np.float32)
    ret = rng.standard_normal((T, N)).astype(np.float32)
    return SimpleNamespace(case=case, desc=desc, lay=lay, slices=slices, flat=flat, obs=obs, hx0=hx0, dones=dones, actions=actions,
                           adv=adv, ret=ret, rng=rng, D=D, H=H, Hg=Hg, A=A, T=T, N=N)


@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as Nt
    return Nt.get_context(0)


GRAD_TOL = 2e-5


def check_grad_vs_fp64(ctx, case):
    """Both minibatch forms (idx NULL, permutation slice): 14 gradient tensors, four losses, zero padding and the clip norm
    against float64.  Returns the worst per-tensor gradient error."""
    cid, br, D, H, Hg, A, T, N, opts = case
    x = make_inputs(case)
    B = T * N
    net = reference_network(x)
    logits, values, _ = reference_forward(x, net)
    lsm = torch.log_softmax(logits.detach().reshape(B, A), -1)
    set_old_log_probs(x, lsm.gather(-1, torch.as_tensor(x.actions.reshape(B, 1).astype(np.int64))).squeeze(-1).numpy())
    d = to_device(x)
    adv_norm = "norm" in opts
    Mp = max(1, 3 * B // 8)
    perm = x.rng.permutation(B).astype(np.int32)
    used = torch.zeros(int(x.lay.total), dtype=torch.bool)
    for off, shape in x.slices.values():
        used[off:off + int(np.prod(shape))] = True
    sumsq = torch.zeros(ctx.grad_sumsq_bytes(int(x.lay.total)) // 8 + 1, dtype=torch.float64, device="cuda")
    adam_ws = torch.empty(ctx.clip_adam_workspace_bytes(int(x.lay.total)) // 8 + 1, dtype=torch.float64, device="cuda")
    worst = 0.0
    for rows, M in ((None, B), (perm[:Mp], Mp)):
        den = 2 * M if "den2" in opts else M
        rsel = np.arange(B) if rows is None else rows.astype(np.int64)
        net.zero_grad()
        total, ref_losses = reference_loss(x, logits, values, rsel, adv_norm, den)
        total.backward(retain_graph=True)
        ref = {n: p.grad.numpy() for n, p in net.named_parameters()}
        hyper = make_hyper(M, den, adv_norm, B)
        hyper.grad_sumsq = sumsq.data_ptr()
        ws = torch.empty(ctx.rnn_workspace_bytes(x.desc, T, N, M, True) // 4 + 64, device="cuda")
        grads, losses = device_grad(ctx, x, d, cuda(rows, torch.int32), M, hyper, ws)
        where = f"{cid} M={M}"
        np.testing.assert_allclose(losses.cpu().numpy(), [float(l) for l in ref_losses], rtol=1e-5, atol=1e-6, err_msg=where)
        g = grads.cpu()
        assert float(g[~used].abs().sum()) == 0.0, where
        for n in x.slices:
            off, shape = x.slices[n]
            got = g[off:off + int(np.prod(shape))].numpy().reshape(ref[n].shape)
            e = nerr(got, ref[n])
            worst = max(worst, e)
            assert e <= GRAD_TOL, (where, n, e)
        ref_norm = float(np.sqrt(sum((r.astype(np.float64) ** 2).sum() for r in ref.values())))
        gn = torch.zeros(1, device="cuda")
        z = torch.zeros_like(grads)
        ctx.clip_adam_step(d.P.clone(), grads.clone(), z, z.clone(), hyper, adam_ws, gn)
        torch.cuda.synchronize()
        assert abs(float(gn) - ref_norm) <= GRAD_TOL * ref_norm, (where, float(gn), ref_norm)
    return worst


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_wide_rnn_grad_minibatch_vs_fp64(ctx, case):
    """dppo_rnn_grad_minibatch on the cluster scans: all 14 gradient tensors (2e-5 of each tensor's largest entry), the losses
    (rtol 1e-5), zero padding and the gradient norm of dppo_clip_adam_step against float64 autograd."""
    worst = check_grad_vs_fp64(ctx, case)
    print(f"{case[0]}: worst gradient error {worst:.2e}")


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_wide_rnn_forward_vs_fp64(ctx, case):
    """dppo_rnn_forward with heads 1, 2 and 3, with the case's resets and initial state and with neither: logits, values and the
    final hidden state agree with float64 to 1e-5."""
    cid, br, D, H, Hg, A, T, N, opts = case
    x = make_inputs(case, seed=1)
    net = reference_network(x)
    ws = torch.empty(ctx.rnn_workspace_bytes(x.desc, T, N, T * N, False) // 4 + 64, device="cuda")
    P, obs = cuda(x.flat), cuda(x.obs)
    tol = lambda ref: 1e-5 * max(1.0, float(np.abs(ref).max()))
    for with_state in (True, False):
        with torch.no_grad():
            rl, rv, rh = (t.numpy() for t in reference_forward(x, net, with_state))
        pd = cuda(x.dones, torch.uint8) if with_state else None
        hx0 = cuda(x.hx0) if with_state else None
        for heads in (1, 2, 3):
            logits = torch.full((T, N, A), float("nan"), device="cuda") if heads & 1 else None
            values = torch.full((T, N), float("nan"), device="cuda") if heads & 2 else None
            hx = torch.full((N, Hg), float("nan"), device="cuda")
            ctx.rnn_forward(x.desc, P, obs, pd, hx0, T, N, heads, logits, values, hx, ws)
            torch.cuda.synchronize()
            where = (cid, with_state, heads)
            if heads & 1:
                assert np.abs(logits.cpu().numpy() - rl).max() <= tol(rl), where
            if heads & 2:
                assert np.abs(values.cpu().numpy() - rv).max() <= tol(rv), where
            assert np.abs(hx.cpu().numpy() - rh[0]).max() <= tol(rh), where


def random_params(desc, lay, rng):
    from diamond.recurrent import rnn_param_slices
    flat = np.zeros(int(lay.total), np.float32)
    for name, (off, shape) in rnn_param_slices(desc, lay).items():
        s = 1.0 / np.sqrt(shape[1]) if len(shape) == 2 else 0.3
        flat[off:off + int(np.prod(shape))] = (rng.standard_normal(int(np.prod(shape))) * s).astype(np.float32)
    return flat


@gpu
def test_wide_rnn_results_do_not_depend_on_env_count(ctx):
    """The same 19 environments inside N = 19, 161 and 577 at Hg = 256 (cluster scans with 2 / 10 / 32 environments per cluster and
    E = 1 / 2 / 4 environments per thread, so the environments land in different clusters and slots): logits, values and the final
    hidden state are bit-identical.  The gradient of a minibatch made of exactly those environments' rows agrees to 1e-6 of each
    tensor's largest entry; it is not bit-identical because the split-K weight-gradient and bias reductions group rows by T * N
    (and by cluster), which changes the order of the fp32 partial sums."""
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    D, H, Hg, A, T, n0 = 5, 64, 256, 4, 9, 19
    desc = Nt.RnnDesc(D, H, Hg, A)
    lay = Nt.rnn_layout(desc)
    rng = np.random.default_rng(256)
    P = cuda(random_params(desc, lay, rng))
    Nmax = 577
    obs = rng.standard_normal((T, Nmax, D)).astype(np.float32)
    dones = rng.random((T, Nmax)) < 0.15
    hx0 = (0.5 * rng.standard_normal((Nmax, Hg))).astype(np.float32)
    actions = rng.integers(0, A, (T, Nmax)).astype(np.int32)
    old_lp = (rng.standard_normal((T, Nmax)) * 0.3 - 1.4).astype(np.float32)
    adv, ret = rng.standard_normal((T, Nmax)).astype(np.float32), rng.standard_normal((T, Nmax)).astype(np.float32)
    out, grads = {}, {}
    for N in (19, 161, 577):
        assert branch(N, Hg) == {19: "c8e1", 161: "c8e2", 577: "c8e4"}[N]
        ws = torch.empty(ctx.rnn_workspace_bytes(desc, T, N, T * N, False) // 4 + 64, device="cuda")
        logits, values, hx = torch.empty(T, N, A, device="cuda"), torch.empty(T, N, device="cuda"), torch.empty(N, Hg, device="cuda")
        o, pd, h0 = cuda(obs[:, :N]), cuda(dones[:, :N], torch.uint8), cuda(hx0[:N])
        ctx.rnn_forward(desc, P, o, pd, h0, T, N, 3, logits, values, hx, ws)
        torch.cuda.synchronize()
        out[N] = (logits[:, :n0].cpu(), values[:, :n0].cpu(), hx[:n0].cpu())
        rows = (np.arange(T)[:, None] * N + np.arange(n0)[None, :]).reshape(-1).astype(np.int32)
        M = rows.size
        hyper = make_hyper(M, M, False, T * N)
        wsg = torch.empty(ctx.rnn_workspace_bytes(desc, T, N, M, True) // 4 + 64, device="cuda")
        g, losses = torch.zeros(int(lay.total), device="cuda"), torch.zeros(4, device="cuda")
        ctx.rnn_grad_minibatch(desc, P, g, o, pd, h0, T, N, cuda(actions[:, :N].reshape(-1), torch.int32),
                               cuda(old_lp[:, :N].reshape(-1)), cuda(adv[:, :N].reshape(-1)), cuda(ret[:, :N].reshape(-1)), None,
                               cuda(rows, torch.int32), M, hyper, losses, wsg)
        torch.cuda.synchronize()
        grads[N] = (g.cpu().double(), losses.cpu().double())
    for N in (161, 577):
        for k, what in enumerate(("logits", "values", "hx_out")):
            assert torch.equal(out[N][k], out[19][k]), (N, what, float((out[N][k] - out[19][k]).abs().max()))
        for name, (off, shape) in rnn_param_slices(desc, lay).items():
            n = int(np.prod(shape))
            ref = grads[19][0][off:off + n]
            err = float((grads[N][0][off:off + n] - ref).abs().max())
            assert err <= 1e-6 * float(ref.abs().max()), (N, name, err)
        assert torch.allclose(grads[N][1], grads[19][1], rtol=1e-6, atol=0)


@gpu
def test_wide_rnn_gradient_additive_and_reproducible(ctx):
    """N = 1024, T = 128, Hg = 256 (32 environments per 8-CTA cluster, E = 4): a repeated call is bit-identical, and with a fixed
    loss denominator the gradients and losses of the two halves of a minibatch add up to those of the whole."""
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    D, H, Hg, A, T, N = 8, 64, 256, 4, 128, 1024
    B, M = T * N, T * N // 8
    assert branch(N, Hg) == "c8e4"
    desc = Nt.RnnDesc(D, H, Hg, A)
    lay = Nt.rnn_layout(desc)
    slices = rnn_param_slices(desc, lay)
    g = torch.Generator(device="cuda").manual_seed(9)
    P = torch.zeros(int(lay.total), device="cuda")
    for name, (off, shape) in slices.items():
        s = 1.0 / np.sqrt(shape[1]) if len(shape) == 2 else 0.3
        P[off:off + int(np.prod(shape))] = torch.randn(int(np.prod(shape)), device="cuda", generator=g) * s
    obs = torch.randn(T, N, D, device="cuda", generator=g)
    pd = (torch.rand(T, N, device="cuda", generator=g) < 0.02).to(torch.uint8)
    hx0 = 0.5 * torch.randn(N, Hg, device="cuda", generator=g)
    actions = torch.randint(0, A, (B,), device="cuda", generator=g, dtype=torch.int32)
    old_lp = torch.randn(B, device="cuda", generator=g) * 0.3 - 1.4
    adv, ret = torch.randn(B, device="cuda", generator=g), torch.randn(B, device="cuda", generator=g)
    idx = torch.randperm(B, device="cuda", generator=g)[:M].to(torch.int32)
    hyper = make_hyper(M, M, False, B)
    ws = torch.empty(ctx.rnn_workspace_bytes(desc, T, N, M, True) // 4 + 64, device="cuda")

    def run(rows):
        grads, losses = torch.zeros(int(lay.total), device="cuda"), torch.zeros(4, device="cuda")
        ctx.rnn_grad_minibatch(desc, P, grads, obs, pd, hx0, T, N, actions, old_lp, adv, ret, None, rows.contiguous(), rows.numel(),
                               hyper, losses, ws)
        torch.cuda.synchronize()
        return grads.double(), losses.double()

    g_all, l_all = run(idx)
    g_again, l_again = run(idx)
    assert torch.equal(g_all, g_again) and torch.equal(l_all, l_again)
    g_a, l_a = run(idx[:M // 2])
    g_b, l_b = run(idx[M // 2:])
    for name, (off, shape) in slices.items():
        n = int(np.prod(shape))
        ref = g_all[off:off + n]
        assert float(ref.abs().max()) > 0, name
        err = float((g_a[off:off + n] + g_b[off:off + n] - ref).abs().max())
        assert err <= 2e-5 * float(ref.abs().max()), (name, err)
    assert torch.allclose(l_a[:3] + l_b[:3], l_all[:3], rtol=1e-5, atol=1e-7)


@gpu
def test_gru_wider_than_512_is_refused(ctx):
    """Hg = 513 is refused with NativeError naming 512 (nothing is launched), and the same context then computes a correct Hg = 256
    gradient."""
    from diamond import _native as Nt
    desc = Nt.RnnDesc(4, 64, 513, 3)
    lay = Nt.rnn_layout(desc)
    T, N = 2, 3
    P = torch.zeros(int(lay.total), device="cuda")
    ws = torch.empty(ctx.rnn_workspace_bytes(desc, T, N, T * N, False) // 4 + 64, device="cuda")
    with pytest.raises(Nt.NativeError, match="512"):
        ctx.rnn_forward(desc, P, torch.zeros(T, N, 4, device="cuda"), None, None, T, N, 3, torch.empty(T, N, 3, device="cuda"),
                        torch.empty(T, N, device="cuda"), torch.empty(N, 513, device="cuda"), ws)
    check_grad_vs_fp64(ctx, CASES[CASE_IDS.index("hg256")])


# ---------------------------------------------------------------- agent level -------------------------------------------------
@gpu
@pytest.mark.parametrize("Hg,N_,T", [(256, 38, 19), (512, 19, 12)])
def test_wide_recurrent_fused_engine_matches_autograd_engine(Hg, N_, T):
    """RecurrentPPO at gru_hidden_dim 256 / 512 runs the fused engine; one learn() (2 epochs, 2 minibatches) equals the same network
    run under torch autograd (RecurrentEngine) on the same rollout: parameters and losses within 1e-4."""
    from diamond import RecurrentPPO, RecurrentPPOConfig, envs
    from diamond.recurrent import RecurrentActorCriticNetwork, RecurrentRollout, FusedRecurrentEngine, RecurrentEngine

    class Same(RecurrentActorCriticNetwork):
        pass

    D, A, H = 6, 3, 64
    agents = []
    for cls in (RecurrentActorCriticNetwork, Same):
        cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, num_epochs=2, num_minibatches=2, verbose=False, network_hidden_dim=H,
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


@gpu
def test_wide_recurrent_device_rollout_graph_replay_and_module():
    """Device CartPole rollout at Hg = 256 (one-step cluster scans, the hidden state ping-ponging between two buffers over an odd
    T): the CUDA-graph replay records exactly what the eager launches record, and the recorded values and log-probs are what the
    torch module computes in float64 from the recorded sequence, to 1e-5."""
    from diamond import RecurrentPPO, RecurrentPPOConfig
    from diamond.envs import DeviceVectorEnv
    N_, T, Hg = 48, 17, 256
    recs = []
    for use_graphs in (True, False):
        cfg = RecurrentPPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=6, total_steps=N_ * T * 100, gru_hidden_dim=Hg)
        agent = RecurrentPPO(DeviceVectorEnv.factory("CartPole-v1", seed=6), cfg)
        agent.engine.use_graphs = use_graphs
        agent.ticker = None
        agent.current_observations, _ = agent.envs.reset(seed=6)
        agent.prev_dones = np.zeros(N_, dtype=bool)
        agent.current_hx = torch.zeros(1, N_, Hg, device=agent.device)
        out = []
        for _ in range(5):
            ro = agent.rollout()
            out.append([getattr(ro, k).clone() for k in ("obs", "actions", "rewards", "terminations", "truncations", "prev_dones", "log_probs",
                                                         "values", "next_values", "hx0")])
        torch.cuda.synchronize()
        if use_graphs:
            assert agent._ro_graph is not None, "graph path was not taken"
            net64 = agent.network.double().cpu()
        recs.append(out)
    for a, b in zip(*recs):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    for obs, actions, rew, term, trunc, prev_dones, log_probs, values, next_values, hx0 in recs[0]:
        with torch.inference_mode():
            logits, v, _ = net64.get_logits_values_and_hx(obs.double().cpu(), hx0.double().cpu(), prev_dones.cpu())
        lp = torch.distributions.Categorical(logits=logits).log_prob(actions.cpu())
        assert float((v - values.cpu().double()).abs().max()) <= 1e-5
        assert float((lp - log_probs.cpu().double()).abs().max()) <= 1e-5
        assert bool(torch.isfinite(next_values).all())
