"""The recurrent kernels (csrc/rnn.cu: dppo_rnn_forward, dppo_rnn_grad_minibatch) through the C ABI against a float64 CPU
autograd reference, on every GRU scan branch.

The reference is diamond.recurrent.RecurrentActorCriticNetwork in float64 on the CPU, loaded from the same flat fp32 parameter
buffer, with the PPO loss written out as in oracle/ppo_oracle.py loss_and_grads.  The gradient is compared tensor by tensor
before any optimiser step: Adam's update m / (sqrt(v) + eps) hardly moves when one tensor's gradient is scaled by a constant, so
comparisons of parameters after Adam steps cannot see a gradient that is off by a constant factor.

The scan kernel is picked from the GRU width Hg and the environment count N (rnn.cu launch_scan_fwd / launch_scan_bwd); the
mirror below restates that choice so that the case table can name, and a CPU test can check, the branch each case runs."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

CLIP, VW, BETA = 0.2, 0.5, 0.01


# ---------------------------------------------------------------- mirror of the scan-branch choice in csrc/rnn.cu ----------
def warp_scan_ok(Hg):                                   # rnn.cu warp_scan_ok
    return Hg in (8, 16, 32)


def tiled_scan_ok(Hg):                                  # rnn.cu tiled_scan_ok
    return Hg % 4 == 0 and 12 <= Hg <= 128


def tiled_scan_E(N, Hg):                                # rnn.cu tiled_scan_E: environments per thread of the tiled kernels
    warps, want = N * Hg // 32, 12 * 148
    return 4 if warps // 4 >= want else 2 if warps // 2 >= want else 1


def tiled_scan_groups(N, Hg, E):                        # rnn.cu tiled_scan_groups
    return min(max(1, 256 // Hg), (N + E - 1) // E)


def scan_branch(N, Hg):
    """The forward / backward scan kernel pair rnn.cu launches for (N, Hg)."""
    if warp_scan_ok(Hg):
        return f"warp{Hg}"
    if tiled_scan_ok(Hg):
        return f"tiled{tiled_scan_E(N, Hg)}"
    return "smem"


def envs_per_block(N, Hg):
    """Environments one scan block owns (rnn.cu scan_blocks)."""
    if warp_scan_ok(Hg):
        return 128 // Hg
    if tiled_scan_ok(Hg):
        E = tiled_scan_E(N, Hg)
        return tiled_scan_groups(N, Hg, E) * E
    return max(1, 256 // Hg)


ALL_BRANCHES = {"warp8", "warp16", "warp32", "tiled1", "tiled2", "tiled4", "smem"}

# One row per case: the branch it is meant to run, then the shapes.  N is one environment past a block boundary wherever the
# branch allows it (last block with a single live environment); H = 128 with A <= 4 takes the role-split head kernel
# (heads.cu head_train_split_kernel), every other (H, A) the generic one.  opts: "hx0" non-zero initial state, "dones" resets
# (else prev_dones NULL), "norm" advantage_norm from fp64 statistics, "den2" loss denominator 2 M (what data parallelism
# passes).
CASES = [
    # id          branch     D    H   Hg  A   T     N   opts
    ("hg1",       "smem",    3,  32,   1, 5, 33,  257, "hx0 dones"),
    ("hg6",       "smem",    4,  32,   6, 5, 64,   43, "hx0 dones norm"),
    ("hg8",       "warp8",   5, 128,   8, 3, 64,   17, "hx0 dones"),
    ("hg10",      "smem",    3, 200,  10, 5,  2,   26, "dones den2"),
    ("hg12",      "tiled1",  6,  64,  12, 4, 33,   22, "hx0 dones"),
    ("hg16",      "warp16",  4, 128,  16, 4, 64,    9, "hx0 dones norm"),
    ("hg16-null", "warp16",  4,  32,  16, 5, 33,   40, ""),
    ("hg32",      "warp32",  8,  32,  32, 5, 33,    5, "hx0 dones den2"),
    ("hg33",      "smem",    5,  64,  33, 2, 17,    8, "hx0 dones"),
    ("hg50",      "smem",    6, 200,  50, 5, 33,    6, "hx0 dones norm"),
    ("hg64",      "tiled1",  8,  64,  64, 4, 33,    5, "hx0 dones"),
    ("hg64-e2",   "tiled2",  8,  64,  64, 4,  3, 1801, "hx0 dones norm"),
    ("hg64-e4",   "tiled4",  8, 128,  64, 4,  4, 4099, "hx0 dones"),
    ("hg127",     "smem",    4,  32, 127, 5,  1,    3, "hx0 dones"),
    ("hg128",     "tiled1",  4, 128, 128, 3,  2,    3, "hx0 dones den2"),
    ("hg128-e4",  "tiled4",  4,  64, 128, 6,  3, 1801, "hx0 dones"),
]
CASE_IDS = [c[0] for c in CASES]


def test_case_table_covers_every_scan_branch():
    """CPU: each case runs the branch it names, and together they run all seven scan kernel pairs, both head kernels and the
    step counts that matter (1: the device rollout's single-step call; 2; an odd count; 64)."""
    seen = set()
    for cid, branch, D, H, Hg, A, T, N, opts in CASES:
        assert scan_branch(N, Hg) == branch, cid
        seen.add(branch)
    assert seen == ALL_BRANCHES
    # E = 2 / 4 at the shapes the existing agent-level tests use, and at Hg = 128
    assert scan_branch(1801, 64) == "tiled2" and scan_branch(4099, 64) == "tiled4" and scan_branch(1800, 128) == "tiled4"
    assert scan_branch(4096, 64) == "tiled4" and scan_branch(64, 64) == "tiled1"
    # every branch has a case whose last scan block holds exactly one environment
    one_past = {b for _, b, D, H, Hg, A, T, N, _ in CASES if N % envs_per_block(N, Hg) == 1}
    assert one_past == ALL_BRANCHES
    assert {1, 2, 64} <= {c[6] for c in CASES} and any(c[6] % 2 == 1 and c[6] > 16 for c in CASES)
    split = [(H, A) for _, _, D, H, Hg, A, T, N, _ in CASES if H == 128 and A <= 4]
    generic = [(H, A) for _, _, D, H, Hg, A, T, N, _ in CASES if not (H == 128 and A <= 4)]
    assert split and any(H == 200 for H, _ in generic) and any(H == 32 for H, _ in generic)


# ---------------------------------------------------------------- inputs and the float64 reference -----------------------------
def make_inputs(case, seed=0):
    cid, branch, D, H, Hg, A, T, N, opts = case
    rng = np.random.default_rng(1000 * CASE_IDS.index(cid) + seed)
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    desc = Nt.RnnDesc(D, H, Hg, A)
    lay = Nt.rnn_layout(desc)
    slices = rnn_param_slices(desc, lay)
    flat = np.zeros(int(lay.total), np.float32)
    for name, (off, shape) in slices.items():
        if len(shape) == 2:
            w = rng.standard_normal(shape) / np.sqrt(shape[1])           # N(0, 1) / sqrt(fan_in)
        else:
            w = 0.3 * rng.standard_normal(shape)
        flat[off:off + int(np.prod(shape))] = w.reshape(-1)
    obs = rng.standard_normal((T, N, D)).astype(np.float32)
    hx0 = (0.5 * rng.standard_normal((N, Hg))).astype(np.float32) if "hx0" in opts else None
    dones = None
    if "dones" in opts:
        dones = rng.random((T, N)) < 0.15
        dones[np.arange(T), rng.integers(0, N, T)] = True                # at least one environment resets at every step
        dones[0, : max(1, N // 3)] = True                                # a block of resets at t = 0 (hx0 discarded)
    actions = rng.integers(0, A, (T, N)).astype(np.int32)
    adv = rng.standard_normal((T, N)).astype(np.float32)
    ret = rng.standard_normal((T, N)).astype(np.float32)
    return SimpleNamespace(case=case, desc=desc, lay=lay, slices=slices, flat=flat, obs=obs, hx0=hx0, dones=dones, actions=actions,
                           adv=adv, ret=ret, rng=rng, D=D, H=H, Hg=Hg, A=A, T=T, N=N)


def reference_network(x):
    """RecurrentActorCriticNetwork in float64 on the CPU with the parameters of the flat fp32 buffer."""
    from diamond.config import RecurrentPPOConfig
    from diamond.recurrent import RecurrentActorCriticNetwork
    cfg = RecurrentPPOConfig(network_hidden_dim=x.H, gru_hidden_dim=x.Hg)
    net = RecurrentActorCriticNetwork(SimpleNamespace(shape=(x.D,)), SimpleNamespace(n=x.A), cfg).double()
    params = dict(net.named_parameters())
    assert set(params) == set(x.slices)
    with torch.no_grad():
        for name, (off, shape) in x.slices.items():
            params[name].copy_(torch.as_tensor(x.flat[off:off + int(np.prod(shape))].astype(np.float64)).reshape(shape))
    return net


def reference_forward(x, net, with_state=True):
    obs = torch.as_tensor(x.obs, dtype=torch.float64)
    hx = torch.as_tensor(x.hx0, dtype=torch.float64).unsqueeze(0) if (with_state and x.hx0 is not None) else None
    dn = torch.as_tensor(x.dones) if (with_state and x.dones is not None) else None
    return net.get_logits_values_and_hx(obs, hx, dn)


def set_old_log_probs(x, new_lp):
    """old log-probs from the fp64 new ones, so that every ratio sits at least 1e-2 from the clip edges 1 -/+ CLIP: half the rows
    in range, a quarter clipped below, a quarter above (both signs of the advantage occur in each group).  A row whose fp32 ratio
    fell on the other side of an edge than its fp64 ratio would change the gradient by ~1/M and fail for the wrong reason."""
    B = new_lp.size
    u = x.rng.random(B)
    ratio = np.where(u < 0.5, x.rng.uniform(1 - CLIP + 0.01, 1 + CLIP - 0.01, B),
                     np.where(u < 0.75, x.rng.uniform(0.5, 1 - CLIP - 0.01, B), x.rng.uniform(1 + CLIP + 0.01, 1.6, B)))
    x.old_lp = (new_lp - np.log(ratio)).astype(np.float32)
    lr = new_lp - x.old_lp.astype(np.float64)                            # the ratio the fp32 old log-prob actually gives
    edge = np.minimum(np.abs(np.exp(lr) - (1 - CLIP)), np.abs(np.exp(lr) - (1 + CLIP)))
    assert edge.min() >= 1e-3


def reference_loss(x, logits, values, rows, adv_norm, den):
    """PPO loss of recurrent_ppo.py:343-359 on the rows `rows` of the flattened [T*N] outputs (oracle/ppo_oracle.py
    loss_and_grads), in float64.  Returns (total, [policy, value, entropy, total])."""
    B, A = x.T * x.N, x.A
    lg = logits.reshape(B, A)[rows]
    v = values.reshape(B)[rows]
    act = torch.as_tensor(x.actions.reshape(B)[rows].astype(np.int64))
    old = torch.as_tensor(x.old_lp[rows].astype(np.float64))
    a = torch.as_tensor(x.adv.reshape(B).astype(np.float64))
    if adv_norm:                                                         # heads.cu adv_norm_consts: fp64 stats, unbiased, + 1e-6
        mu = a.mean()
        a = (a - mu) / (torch.sqrt(((a - mu) ** 2).sum() / (B - 1)) + 1e-6)
    a = a[rows]
    ret = torch.as_tensor(x.ret.reshape(B)[rows].astype(np.float64))
    lsm = torch.log_softmax(lg, -1)
    ratio = torch.exp(lsm.gather(-1, act.unsqueeze(-1)).squeeze(-1) - old)
    pol = torch.max(-a * ratio, -a * torch.clamp(ratio, 1 - CLIP, 1 + CLIP)).sum() / den
    val = 0.5 * ((v - ret) ** 2).sum() / den
    ent = (-(lsm.exp() * lsm).sum(-1)).sum() / den
    total = pol + VW * val - BETA * ent
    return total, [pol, val, ent, total]


# ---------------------------------------------------------------- device side -------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as Nt
    return Nt.get_context(0)


def cuda(a, dtype=torch.float32):
    return None if a is None else torch.as_tensor(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype).contiguous()


def nerr(a, ref):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(a - ref).max() / max(np.abs(ref).max(), 1e-30)


def make_hyper(M, den, adv_norm, adv_count):
    from diamond import _native as Nt
    h = Nt.Hyper()
    h.ppo_clip, h.value_loss_weight, h.entropy_beta = CLIP, VW, BETA
    h.grad_norm_clip, h.adam_eps, h.lr = 0.5, 1e-5, 3e-4
    h.beta1, h.beta2, h.step = 0.9, 0.999, 1
    h.advantage_norm, h.adv_count, h.loss_denominator = int(adv_norm), adv_count, den
    return h


def device_grad(ctx, x, d, idx, M, hyper, ws):
    """One dppo_rnn_grad_minibatch call: (flat gradient, losses) on the host; grads starts filled with 7.0."""
    grads = torch.full((int(x.lay.total),), 7.0, device="cuda")
    losses = torch.zeros(4, device="cuda")
    ctx.rnn_grad_minibatch(x.desc, d.P, grads, d.obs, d.pd, d.hx0, x.T, x.N, d.actions, d.old_lp, d.adv, d.ret, d.stats, idx, M,
                           hyper, losses, ws)
    torch.cuda.synchronize()
    return grads, losses


def to_device(x):
    B = x.T * x.N
    a64 = x.adv.astype(np.float64).reshape(-1)
    return SimpleNamespace(P=cuda(x.flat), obs=cuda(x.obs), pd=cuda(x.dones, torch.uint8), hx0=cuda(x.hx0),
                           actions=cuda(x.actions.reshape(B), torch.int32), old_lp=cuda(x.old_lp), adv=cuda(x.adv.reshape(B)),
                           ret=cuda(x.ret.reshape(B)), stats=cuda(np.array([a64.sum(), (a64 ** 2).sum()]), torch.float64))


# Gradient bar: per-tensor infinity norm relative to the tensor's largest entry (the MLP gradient test's bar).
GRAD_TOL = 2e-5


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_rnn_grad_minibatch_vs_fp64(ctx, case):
    """The flat gradient (all 14 tensors), the four losses and the gradient norm handed to the clip, for the whole rollout as one
    minibatch (idx NULL) and for a permutation slice of it (rows scattered back before the backward scan), against float64
    autograd.  Padding between the tensors comes out zero."""
    cid, branch, D, H, Hg, A, T, N, opts = case
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
    names = list(x.slices)
    used = torch.zeros(int(x.lay.total), dtype=torch.bool)
    for off, shape in x.slices.values():
        used[off:off + int(np.prod(shape))] = True
    sumsq = torch.zeros(ctx.grad_sumsq_bytes(int(x.lay.total)) // 8 + 1, dtype=torch.float64, device="cuda")
    adam_ws = torch.empty(ctx.clip_adam_workspace_bytes(int(x.lay.total)) // 8 + 1, dtype=torch.float64, device="cuda")
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
        for n in names:
            off, shape = x.slices[n]
            got = g[off:off + int(np.prod(shape))].numpy().reshape(ref[n].shape)
            assert nerr(got, ref[n]) <= GRAD_TOL, (where, n, nerr(got, ref[n]))
        # the norm dppo_clip_adam_step clips with: from the fp64 partial sums the gradient assembly left in hyper.grad_sumsq, and
        # from its own norm kernel (hyper.grad_sumsq NULL); both against the fp64 norm of the reference gradient
        ref_norm = float(np.sqrt(sum((r.astype(np.float64) ** 2).sum() for r in ref.values())))
        norms = []
        for fused in (True, False):
            hyper.grad_sumsq = sumsq.data_ptr() if fused else None
            gn = torch.zeros(1, device="cuda")
            z = torch.zeros_like(grads)
            ctx.clip_adam_step(d.P.clone(), grads.clone(), z, z.clone(), hyper, adam_ws, gn)
            torch.cuda.synchronize()
            norms.append(float(gn))
        assert abs(norms[0] - ref_norm) <= GRAD_TOL * ref_norm, (where, norms[0], ref_norm)
        assert abs(norms[0] - norms[1]) <= 1e-6 * ref_norm, (where, norms)


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_rnn_forward_vs_fp64(ctx, case):
    """dppo_rnn_forward: logits, values and the final hidden state for heads 1 (actor), 2 (critic) and 3, with the case's resets and
    initial state and with both NULL (no resets, zero state), against float64."""
    cid, branch, D, H, Hg, A, T, N, opts = case
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


@gpu
def test_rnn_results_do_not_depend_on_env_count(ctx):
    """The same 64 environments inside N = 64, 1801 and 4099 environments at Hg = 64, which run the tiled scans with E = 1, 2 and 4
    environments per thread: logits, values and the final hidden state are bit-identical.  The tiled kernels keep one summation order (rnn.cu), and so do the launches around them: the base and
    input-projection GEMMs (gemm_simt.cu; the 128- and 64-row tile configurations both run one k-ascending FMA chain per output)
    and the head kernels (one warp per row)."""
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    D, H, Hg, A, T = 8, 64, 64, 4, 8
    desc = Nt.RnnDesc(D, H, Hg, A)
    lay = Nt.rnn_layout(desc)
    rng = np.random.default_rng(64)
    flat = np.zeros(int(lay.total), np.float32)
    for name, (off, shape) in rnn_param_slices(desc, lay).items():
        s = 1.0 / np.sqrt(shape[1]) if len(shape) == 2 else 0.3
        flat[off:off + int(np.prod(shape))] = (rng.standard_normal(int(np.prod(shape))) * s).astype(np.float32)
    P = cuda(flat)
    Nmax = 4099
    obs = rng.standard_normal((T, Nmax, D)).astype(np.float32)
    dones = rng.random((T, Nmax)) < 0.15
    hx0 = (0.5 * rng.standard_normal((Nmax, Hg))).astype(np.float32)
    out = {}
    for N in (64, 1801, 4099):
        assert scan_branch(N, Hg) == {64: "tiled1", 1801: "tiled2", 4099: "tiled4"}[N]
        ws = torch.empty(ctx.rnn_workspace_bytes(desc, T, N, T * N, False) // 4 + 64, device="cuda")
        logits, values, hx = torch.empty(T, N, A, device="cuda"), torch.empty(T, N, device="cuda"), torch.empty(N, Hg, device="cuda")
        ctx.rnn_forward(desc, P, cuda(obs[:, :N]), cuda(dones[:, :N], torch.uint8), cuda(hx0[:N]), T, N, 3, logits, values, hx, ws)
        torch.cuda.synchronize()
        out[N] = (logits[:, :64].cpu(), values[:, :64].cpu(), hx[:64].cpu())
    for N in (1801, 4099):
        for k, what in enumerate(("logits", "values", "hx_out")):
            assert torch.equal(out[N][k], out[64][k]), (N, what, float((out[N][k] - out[64][k]).abs().max()))


@gpu
def test_rnn_gradient_additive_and_reproducible_at_full_size(ctx):
    """At the measured RecurrentPPO scale (T = 128, N = 4096, Hg = 64: the E = 4 tiled scans, a 65 536-row minibatch): a repeated
    call is bit-identical, and with a fixed loss denominator the gradients and losses of the two halves of the minibatch add up
    to those of the whole."""
    from diamond import _native as Nt
    from diamond.recurrent import rnn_param_slices
    D, H, Hg, A, T, N = 8, 64, 64, 4, 128, 4096
    B, M = T * N, T * N // 8
    assert scan_branch(N, Hg) == "tiled4"
    desc = Nt.RnnDesc(D, H, Hg, A)
    lay = Nt.rnn_layout(desc)
    slices = rnn_param_slices(desc, lay)
    g = torch.Generator(device="cuda").manual_seed(7)
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
