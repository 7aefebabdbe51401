"""GPU: each CUDA kernel, called through the C ABI, against the CPU oracle on identical inputs."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ppo_oracle as O
from oracle import c_oracle as CO

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
GAE_CASES = ["kat1", "kat2", "rand_small", "rand_ragged", "rand_mid", "t1", "both_masks"]


@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as N
    return N.get_context(0)


def dev(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x)).to(device="cuda", dtype=dtype).contiguous()


def nerr(a, ref):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(a - ref).max() / max(np.abs(ref).max(), 1e-30)


# ---------------------------------------------------------------- GAE -------------------------
@pytest.mark.parametrize("case", GAE_CASES)
@pytest.mark.parametrize("tag,gam,lam", [("", 0.99, 0.95), (".g9l8", 0.9, 0.8)])
def test_gae_golden(ctx, case, tag, gam, lam):
    g = np.load(os.path.join(GOLDEN, "gae.npz"))
    args = [dev(g[f"{case}.{k}"]) for k in ("rewards", "terminations", "truncations", "values", "next_values")]
    ret = torch.empty_like(args[0])
    stats = torch.zeros(2, dtype=torch.float64, device="cuda")
    adv = ctx.gae(*args, gam, lam, returns=ret, stats=stats)
    ref = g[f"{case}{tag}.advantages"]
    # tolerance of BASELINE.json north_star: 1e-5 relative, normalised (SURVEY §8d)
    assert nerr(adv.cpu().numpy(), ref) <= 1e-5
    np.testing.assert_allclose(adv.cpu().numpy(), ref, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ret.cpu().numpy(), g[f"{case}.values"] + ref, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(stats.cpu().numpy(), [ref.astype(np.float64).sum(), (ref.astype(np.float64) ** 2).sum()],
                               rtol=1e-5, atol=1e-5)
    if tag == "" and f"{case}.adv_norm" in g:
        an = ctx.adv_normalize(adv, stats, adv.numel())
        refn = g[f"{case}.adv_norm"]
        assert np.abs(an.cpu().numpy() - refn).max() <= 2e-5 * max(1.0, np.abs(refn).max())


def test_gae_known_answer_vectors(ctx):
    """SURVEY §8c KATs: rewards = 1 geometric sums; termination (no bootstrap, trace cut) vs truncation (bootstrap, trace cut)."""
    z = lambda *s: torch.zeros(*s, device="cuda")
    adv = ctx.gae(torch.ones(8, 1, device="cuda"), z(8, 1), z(8, 1), z(8, 1), z(8, 1), 0.99, 0.95).cpu().numpy()[:, 0]
    np.testing.assert_allclose(adv, [6.5182, 5.8673, 5.1752, 4.4394, 3.6570, 2.8250, 1.9405, 1.0000], atol=5e-5)
    r, v, nv = torch.ones(4, 3, device="cuda"), torch.full((4, 3), 0.5, device="cuda"), torch.full((4, 3), 2.0, device="cuda")
    te, tr = z(4, 3), z(4, 3)
    te[1, 1] = 1.0
    tr[1, 2] = 1.0
    ret = torch.empty(4, 3, device="cuda")
    adv = ctx.gae(r, te, tr, v, nv, 0.99, 0.95, returns=ret).cpu().numpy()
    ref = np.array([[9.069237, 2.950250, 4.812440], [7.006100, 0.500000, 2.480000], [4.812440] * 3, [2.480000] * 3])
    np.testing.assert_allclose(adv, ref, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(ret.cpu().numpy(), ref + 0.5, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("T,N", [(1, 1), (1, 4096), (2, 1), (2048, 3), (129, 4097), (128, 28), (128, 29)])
def test_gae_edge_shapes_vs_c_oracle(ctx, T, N):
    """Single step / single env, sizes straddling the 28-env CTA tile and the 128-step chunking of the pipelined kernel, every
    step finished (all masks set), and no step finished."""
    rng = np.random.default_rng(T * 7 + N)
    r, v, nv = (rng.standard_normal((T, N)).astype(np.float32) for _ in range(3))
    for mode in ("mixed", "all_done", "none"):
        te = {"mixed": (rng.random((T, N)) < 0.3), "all_done": np.ones((T, N), bool), "none": np.zeros((T, N), bool)}[mode].astype(np.float32)
        tr = ((rng.random((T, N)) < 0.3) & (te == 0)).astype(np.float32) if mode == "mixed" else np.zeros((T, N), np.float32)
        ref, _ = CO.gae(r, te, tr, v, nv)
        ret = torch.empty(T, N, device="cuda")
        adv = ctx.gae(dev(r), dev(te), dev(tr), dev(v), dev(nv), 0.99, 0.95, returns=ret).cpu().numpy()
        assert nerr(adv, ref) <= 1e-5, mode
        np.testing.assert_allclose(ret.cpu().numpy(), v + ref, rtol=1e-5, atol=1e-5)


def test_gae_linearity_and_time_locality_at_full_size(ctx):
    """Size-independent properties at BASELINE.json's 4096 x 128: GAE is linear in (rewards, values, next_values) for fixed masks,
    and a finished step cuts the trace -- advantages before a done step do not depend on anything after it."""
    T, N = 128, 4096
    g = torch.Generator(device="cuda").manual_seed(5)
    rnd = lambda: torch.randn(T, N, device="cuda", generator=g)
    te = (torch.rand(T, N, device="cuda", generator=g) < 0.01).float()
    tr = ((torch.rand(T, N, device="cuda", generator=g) < 0.01) & (te == 0)).float()
    r1, v1, n1, r2, v2, n2 = rnd(), rnd(), rnd(), rnd(), rnd(), rnd()
    a1 = ctx.gae(r1, te, tr, v1, n1, 0.99, 0.95)
    a2 = ctx.gae(r2, te, tr, v2, n2, 0.99, 0.95)
    a12 = ctx.gae(r1 + 2 * r2, te, tr, v1 + 2 * v2, n1 + 2 * n2, 0.99, 0.95)
    assert (a12 - (a1 + 2 * a2)).abs().max().item() <= 1e-5 * a12.abs().max().item()
    # cut: make every env finish at step 63; perturbing steps >= 64 must leave steps <= 63 bit-identical
    te2 = te.clone(); te2[63] = 1.0
    base = ctx.gae(r1, te2, tr * (1 - te2), v1, n1, 0.99, 0.95)
    r3, v3, n3 = r1.clone(), v1.clone(), n1.clone()
    r3[64:] += 3.0; v3[64:] -= 1.0; n3[64:] *= 2.0
    pert = ctx.gae(r3, te2, tr * (1 - te2), v3, n3, 0.99, 0.95)
    assert torch.equal(base[:64], pert[:64])
    assert not torch.equal(base[64:], pert[64:])


@pytest.mark.parametrize("T,N", [(128, 4096), (128, 1000), (300, 77), (5, 33), (128, 8)])
def test_gae_random_vs_c_oracle(ctx, T, N):
    rng = np.random.default_rng(T * 1000 + N)
    r = rng.standard_normal((T, N)).astype(np.float32)
    te = (rng.random((T, N)) < 0.01).astype(np.float32)
    tr = ((rng.random((T, N)) < 0.01) & (te == 0)).astype(np.float32)
    v = rng.standard_normal((T, N)).astype(np.float32)
    nv = rng.standard_normal((T, N)).astype(np.float32)
    ref_a, ref_r = CO.gae(r, te, tr, v, nv)
    ret = torch.empty(T, N, device="cuda")
    adv = ctx.gae(dev(r), dev(te), dev(tr), dev(v), dev(nv), 0.99, 0.95, returns=ret)
    assert nerr(adv.cpu().numpy(), ref_a) <= 1e-5
    assert nerr(ret.cpu().numpy(), ref_r) <= 1e-5
    # masks cut the trace exactly: an advantage at a terminated step equals r - v
    a = adv.cpu().numpy()
    np.testing.assert_allclose(a[te == 1], (r - v)[te == 1], rtol=1e-6, atol=1e-6)


# ---------------------------------------------------------------- MLP -------------------------
def rand_params(rng, names, D, H, A, cont, scale=0.3):
    head = "actor_mean_head" if cont else "actor_head"
    shapes = {"base.0.weight": (H, D), "base.0.bias": (H,), "base.2.weight": (H, H), "base.2.bias": (H,),
              f"{head}.0.weight": (H, H), f"{head}.0.bias": (H,), f"{head}.2.weight": (A, H), f"{head}.2.bias": (A,),
              "critic_head.0.weight": (H, H), "critic_head.0.bias": (H,), "critic_head.2.weight": (1, H),
              "critic_head.2.bias": (1,), "actor_log_std": (1, A)}
    p = {}
    for n in names:
        fan_in = shapes[n][-1] if len(shapes[n]) > 1 else 1
        s = scale if len(shapes[n]) == 1 else 1.0 / np.sqrt(fan_in)
        p[n] = torch.as_tensor((rng.standard_normal(shapes[n]) * s).astype(np.float32))
    return p


CONFIGS = [
    # D, H, A, cont, B, M
    (4, 64, 2, False, 1024, 128),
    (8, 64, 4, False, 1024, 128),
    (3, 64, 1, True, 4096, 512),
    (5, 64, 3, True, 512, 128),
    (64, 128, 4, False, 1024, 128),
    (64, 256, 4, False, 8192, 2048),
    (17, 96, 7, False, 700, 333),
    (64, 256, 6, True, 4096, 1500),
    # role-split head kernel (H in {128, 256}, A <= 4): ragged row counts (actor warps take 2 rows, critic warps 4), A < 4, Gaussian
    (64, 256, 3, False, 4096, 1023),
    (64, 256, 3, True, 4096, 1501),
    (16, 128, 2, True, 2048, 1023),
    (16, 128, 1, False, 2048, 7),
    # H = 512: head_train_kernel<16, 4, 1> / head_eval_kernel<16>, a 1024-row discrete minibatch and a Gaussian one
    (32, 512, 4, False, 4096, 1024),
    (6, 512, 9, True, 2048, 700),
    # A = 32 (DPPO_MAX_ACT: every lane of the warp an action) with H not a multiple of 32; (A + 1) * H = 4950 needs 178 KB of
    # shared memory in the head kernel, under its 200 KB bound
    (10, 150, 32, False, 1000, 333),
    (12, 40, 32, True, 700, 255),
]


def f64(p):
    """The oracle is dtype-generic: parameters (and inputs) in float64 make it a float64 reference."""
    return {k: v.double() for k, v in p.items()}


@pytest.mark.parametrize("D,H,A,cont,B,M", CONFIGS)
def test_mlp_forward_and_logprob(ctx, D, H, A, cont, B, M):
    from diamond.flat import FlatMlp
    rng = np.random.default_rng(D * 7 + H)
    names = O.CONTINUOUS_PARAM_NAMES if cont else O.DISCRETE_PARAM_NAMES
    p = rand_params(rng, names, D, H, A, cont)
    fm = FlatMlp(D, H, A, cont)
    flat = fm.pack(p, device="cuda")
    obs = rng.standard_normal((B, D)).astype(np.float32)
    p64 = f64(p)
    ref_out, ref_v = O.mlp_forward(p64, torch.as_tensor(obs).double(), cont)
    ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, 300, False) // 4, device="cuda")      # forces row chunking
    out = torch.empty(B, A, device="cuda"); val = torch.empty(B, device="cuda")
    ctx.mlp_forward(fm.desc, flat, dev(obs), B, 3, out, val, ws)
    assert nerr(out.cpu().numpy(), ref_out.numpy()) <= 1e-5
    assert nerr(val.cpu().numpy(), ref_v.numpy()) <= 1e-5
    # critic-only and gathered rows
    idx = rng.permutation(B)[:M].astype(np.int32)
    val2 = torch.empty(M, device="cuda")
    ctx.mlp_forward(fm.desc, flat, dev(obs), M, 2, None, val2, ws, idx=dev(idx, torch.int32))
    assert nerr(val2.cpu().numpy(), ref_v.numpy()[idx]) <= 1e-5
    lp = torch.empty(B, device="cuda")
    if cont:
        act = rng.standard_normal((B, A)).astype(np.float32)
        ctx.logprob_gaussian(out, flat[fm.layout.log_std:fm.layout.log_std + A], dev(act), lp)
        ref_lp = O.normal_log_prob(ref_out, p64["actor_log_std"].expand_as(ref_out), torch.as_tensor(act).double())
    else:
        act = rng.integers(0, A, B)
        ctx.logprob_categorical(out, dev(act, torch.int32), lp)
        ref_lp, _ = O.categorical_log_prob(ref_out, torch.as_tensor(act))
    np.testing.assert_allclose(lp.cpu().numpy(), ref_lp.numpy(), rtol=1e-4, atol=1e-5)


def make_hyper(N, M, step=1, adv_norm=False, adv_count=0, **kw):
    cfg = O.default_cfg(**kw)
    h = N.Hyper()
    h.ppo_clip, h.value_loss_weight, h.entropy_beta = cfg["ppo_clip"], cfg["value_loss_weight"], cfg["entropy_beta"]
    h.grad_norm_clip, h.adam_eps, h.lr = cfg["grad_norm_clip"], cfg["adam_eps"], cfg["lr"]
    h.beta1, h.beta2, h.step = 0.9, 0.999, step
    h.advantage_norm, h.adv_count, h.loss_denominator = int(adv_norm), adv_count, M
    return h, cfg


@pytest.mark.parametrize("D,H,A,cont,B,M", CONFIGS)
def test_mlp_grad_minibatch_vs_oracle(ctx, D, H, A, cont, B, M):
    from diamond import _native as N
    from diamond.flat import FlatMlp
    rng = np.random.default_rng(D * 13 + H + A)
    names = O.CONTINUOUS_PARAM_NAMES if cont else O.DISCRETE_PARAM_NAMES
    p = rand_params(rng, names, D, H, A, cont)
    fm = FlatMlp(D, H, A, cont)
    flat = fm.pack(p, device="cuda")
    obs = rng.standard_normal((B, D)).astype(np.float32)
    act = rng.standard_normal((B, A)).astype(np.float32) if cont else rng.integers(0, A, B)
    old_lp = (rng.standard_normal(B) * 0.3 - (1.0 if not cont else 1.5 * A)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32)
    ret = rng.standard_normal(B).astype(np.float32)
    idx = rng.permutation(B)[:M].astype(np.int32)
    hyper, cfg = make_hyper(N, M)
    t = lambda a: torch.as_tensor(a).double() if a.dtype.kind == "f" else torch.as_tensor(a)
    sel = torch.as_tensor(idx.astype(np.int64))
    losses_ref, g_ref = O.loss_and_grads(f64(p), t(obs)[sel], t(act)[sel], t(old_lp)[sel], t(adv)[sel], t(ret)[sel], cfg, cont)

    grads = torch.full((fm.total,), 7.0, device="cuda")
    losses = torch.zeros(4, device="cuda")
    ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, M, True) // 4 + 64, device="cuda")
    ctx.mlp_grad_minibatch(fm.desc, flat, grads, dev(obs), dev(act, torch.float32 if cont else torch.int32), dev(old_lp),
                           dev(adv), dev(ret), None, dev(idx, torch.int32), M, hyper, losses, ws)
    torch.cuda.synchronize()
    got = losses.cpu().numpy()
    ref = np.array([losses_ref[k] for k in ("policy", "value", "entropy", "total")])
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-6)
    gv = fm.views(grads)
    for n in names:
        e = nerr(gv[n].cpu().numpy(), g_ref[n].numpy())
        assert e <= 2e-5, (n, e)
    # padding between tensors is zeroed
    used = torch.zeros(fm.total, dtype=torch.bool)
    for n, (off, shape) in fm.slices.items():
        used[off:off + int(np.prod(shape))] = True
    assert float(grads.cpu()[~used].abs().sum()) == 0.0


def test_head_shape_over_the_shared_memory_bound_is_refused(ctx):
    """H = 512 with A = 12 needs (A + 1) * H floats of weights plus per-warp accumulators: over the head kernel's 200 KB of shared
    memory.  The host-side check refuses the launch with NativeError (nothing runs in a broken state), and the context keeps
    working: the next call with a valid shape computes the right gradient."""
    from diamond import _native as N
    from diamond.flat import FlatMlp
    rng = np.random.default_rng(12)
    for D, H, A, ok in ((8, 512, 12, False), (8, 512, 4, True)):
        B = M = 256
        p = rand_params(rng, O.DISCRETE_PARAM_NAMES, D, H, A, False)
        fm = FlatMlp(D, H, A, False)
        obs = rng.standard_normal((B, D)).astype(np.float32)
        act = rng.integers(0, A, B)
        old_lp, adv, ret = (rng.standard_normal(B).astype(np.float32) for _ in range(3))
        hyper, cfg = make_hyper(N, M)
        grads = torch.zeros(fm.total, device="cuda"); losses = torch.zeros(4, device="cuda")
        ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, M, True) // 4 + 64, device="cuda")
        args = (fm.desc, fm.pack(p, device="cuda"), grads, dev(obs), dev(act, torch.int32), dev(old_lp), dev(adv), dev(ret), None,
                dev(np.arange(M), torch.int32), M, hyper, losses, ws)
        if not ok:
            with pytest.raises(N.NativeError, match="too large for shared memory"):
                ctx.mlp_grad_minibatch(*args)
            continue
        ctx.mlp_grad_minibatch(*args)
        torch.cuda.synchronize()
        t = lambda a: torch.as_tensor(a).double() if a.dtype.kind == "f" else torch.as_tensor(a)
        losses_ref, g_ref = O.loss_and_grads(f64(p), t(obs), t(act), t(old_lp), t(adv), t(ret), cfg, False)
        np.testing.assert_allclose(losses.cpu().numpy(), [losses_ref[k] for k in ("policy", "value", "entropy", "total")],
                                   rtol=1e-4, atol=1e-6)
        gv = fm.views(grads)
        for n in O.DISCRETE_PARAM_NAMES:
            assert nerr(gv[n].cpu().numpy(), g_ref[n].numpy()) <= 2e-5, n


def test_update_gradient_is_additive_over_samples_at_full_size(ctx):
    """Size-independent property at BASELINE.json's full minibatch (65 536 rows of the 4096 x 128 buffer, D = 64, 2x256 + heads):
    with a fixed loss denominator the minibatch gradient is the sum of the gradients of its two halves, the losses are the sums of
    the halves' losses, and the result does not depend on the order of the rows (up to fp32 summation order) -- through
    the tensor-core path (tcgen05 GEMMs, joint weight-gradient launch, head kernel, deterministic reduction)."""
    from diamond import _native as N
    from diamond.flat import FlatMlp
    D, H, A, B, M = 64, 256, 4, 524288, 65536
    rng = np.random.default_rng(21)
    p = rand_params(rng, O.DISCRETE_PARAM_NAMES, D, H, A, False)
    fm = FlatMlp(D, H, A, False)
    flat = fm.pack(p, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(2)
    obs = torch.randn(B, D, device="cuda", generator=g)
    act = torch.randint(0, A, (B,), device="cuda", generator=g, dtype=torch.int32)
    old_lp = torch.randn(B, device="cuda", generator=g) * 0.3 - 1.0
    adv, ret = torch.randn(B, device="cuda", generator=g), torch.randn(B, device="cuda", generator=g)
    idx = torch.randperm(B, device="cuda", generator=g)[:M].to(torch.int32)
    hyper, _ = make_hyper(N, M)
    ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, M, True) // 4 + 512, device="cuda")

    def run(rows):
        grads = torch.zeros(fm.total, device="cuda"); losses = torch.zeros(4, device="cuda")
        ctx.mlp_grad_minibatch(fm.desc, flat, grads, obs, act, old_lp, adv, ret, None, rows.contiguous(), rows.numel(), hyper, losses, ws)
        torch.cuda.synchronize()
        return grads.double(), losses.double()

    g_all, l_all = run(idx)
    g_a, l_a = run(idx[:M // 2])
    g_b, l_b = run(idx[M // 2:])
    g_perm, l_perm = run(idx[torch.randperm(M, device="cuda", generator=g)])
    g_again, l_again = run(idx)
    assert torch.equal(g_all, g_again) and torch.equal(l_all, l_again)                   # bit-reproducible
    views = lambda x: fm.views(x)
    for name in O.DISCRETE_PARAM_NAMES:
        ref = views(g_all)[name]
        scale = ref.abs().max().item()
        assert (views(g_a)[name] + views(g_b)[name] - ref).abs().max().item() <= 2e-5 * scale, name
        assert (views(g_perm)[name] - ref).abs().max().item() <= 2e-5 * scale, name
    # policy / value / entropy terms are means over the fixed denominator: halves add up
    assert torch.allclose(l_a[:3] + l_b[:3], l_all[:3], rtol=1e-5, atol=1e-7)
    assert torch.allclose(l_perm, l_all, rtol=1e-5, atol=1e-7)


def test_mlp_grad_advantage_norm_on_the_fly(ctx):
    from diamond import _native as N
    from diamond.flat import FlatMlp
    D, H, A, B, M = 8, 64, 4, 2048, 256
    rng = np.random.default_rng(3)
    p = rand_params(rng, O.DISCRETE_PARAM_NAMES, D, H, A, False)
    fm = FlatMlp(D, H, A, False)
    flat = fm.pack(p, device="cuda")
    obs = rng.standard_normal((B, D)).astype(np.float32)
    act = rng.integers(0, A, B)
    old_lp = (rng.standard_normal(B) * 0.3 - 1.0).astype(np.float32)
    adv = (rng.standard_normal(B) * 3 + 1.5).astype(np.float32)
    ret = rng.standard_normal(B).astype(np.float32)
    idx = rng.permutation(B)[:M].astype(np.int32)
    _, adv_n = O.returns_and_normalise(np.zeros(B, np.float32), adv, True)
    hyper, cfg = make_hyper(N, M, adv_norm=True, adv_count=B)
    t = torch.as_tensor
    sel = t(idx.astype(np.int64))
    losses_ref, g_ref = O.loss_and_grads(p, t(obs)[sel], t(act)[sel], t(old_lp)[sel], t(adv_n)[sel], t(ret)[sel], cfg, False)
    stats = torch.tensor([adv.astype(np.float64).sum(), (adv.astype(np.float64) ** 2).sum()], dtype=torch.float64, device="cuda")
    grads = torch.empty(fm.total, device="cuda"); losses = torch.zeros(4, device="cuda")
    ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, M, True) // 4 + 64, device="cuda")
    ctx.mlp_grad_minibatch(fm.desc, flat, grads, dev(obs), dev(act, torch.int32), dev(old_lp), dev(adv), dev(ret), stats,
                           dev(idx, torch.int32), M, hyper, losses, ws)
    np.testing.assert_allclose(losses.cpu().numpy(), [losses_ref[k] for k in ("policy", "value", "entropy", "total")], rtol=1e-4, atol=1e-6)
    gv = fm.views(grads)
    for n in O.DISCRETE_PARAM_NAMES:
        assert nerr(gv[n].cpu().numpy(), g_ref[n].numpy()) <= 5e-5, n


@pytest.mark.parametrize("n", [13, 12995, 215301])
def test_clip_adam_vs_oracle(ctx, n):
    from diamond import _native as N
    rng = np.random.default_rng(n)
    p0 = rng.standard_normal(n).astype(np.float32)
    names = ["x"]
    p = {"x": torch.as_tensor(p0.copy())}
    state = O.new_adam_state(p, names)
    dp, dm, dv = dev(p0), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    ws = torch.empty(ctx.clip_adam_workspace_bytes(n) // 8 + 1, dtype=torch.float64, device="cuda")
    gn = torch.zeros(1, device="cuda")
    for step in range(1, 6):
        g = (rng.standard_normal(n) * (0.01 if step % 2 else 3.0)).astype(np.float32)
        grads = {"x": torch.as_tensor(g.copy())}
        ref_norm = O.clip_grad_norm_(grads, names, 0.5)
        O.adam_step_(p, grads, state, names, 3e-4, 1e-5)
        hyper, _ = make_hyper(N, 1, step=step)
        dg = dev(g)
        ctx.clip_adam_step(dp, dg, dm, dv, hyper, ws, gn)
        assert abs(float(gn) - ref_norm) <= 1e-5 * ref_norm
        assert nerr(dg.cpu().numpy(), grads["x"].numpy()) <= 1e-5   # torch sums the norm in fp32, the kernel in fp64
    assert nerr(dp.cpu().numpy(), p["x"].numpy()) <= 1e-5
    assert nerr(dm.cpu().numpy(), state["exp_avg"]["x"].numpy()) <= 1e-5
    assert nerr(dv.cpu().numpy(), state["exp_avg_sq"]["x"].numpy()) <= 1e-5


@pytest.mark.parametrize("cont", [False, True])
def test_standalone_loss_vs_oracle(ctx, cont):
    from diamond import _native as N
    M, A = 1000, 5
    rng = np.random.default_rng(5)
    head = torch.as_tensor(rng.standard_normal((M, A)).astype(np.float32), ).requires_grad_(True)
    values = torch.as_tensor(rng.standard_normal(M).astype(np.float32)).requires_grad_(True)
    log_std = torch.as_tensor((rng.standard_normal((1, A)) * 0.2).astype(np.float32)).requires_grad_(True)
    act = rng.standard_normal((M, A)).astype(np.float32) if cont else rng.integers(0, A, M)
    old_lp = (rng.standard_normal(M) * 0.3 - 2).astype(np.float32)
    adv = rng.standard_normal(M).astype(np.float32); ret = rng.standard_normal(M).astype(np.float32)
    # torch-autograd reference of the same loss (what the reference computes for a custom network)
    if cont:
        dist = torch.distributions.Normal(head, log_std.expand_as(head).exp())
        new_lp = dist.log_prob(torch.as_tensor(act)).sum(-1); ent = dist.entropy().sum(-1).mean()
    else:
        dist = torch.distributions.Categorical(logits=head)
        new_lp = dist.log_prob(torch.as_tensor(act)); ent = dist.entropy().mean()
    ratio = (new_lp - torch.as_tensor(old_lp)).exp()
    a = torch.as_tensor(adv)
    lp = torch.max(-a * ratio, -a * torch.clamp(ratio, 0.8, 1.2)).mean()
    lv = 0.5 * torch.nn.functional.mse_loss(values, torch.as_tensor(ret))
    total = lp + 1.0 * lv + -0.01 * ent
    total.backward()
    hyper, _ = make_hyper(N, M)
    ws = torch.empty(ctx.ppo_loss_workspace_bytes(M, A) // 4 + 16, device="cuda")
    losses = torch.zeros(4, device="cuda"); dhead = torch.empty(M, A, device="cuda"); dval = torch.empty(M, device="cuda")
    if cont:
        dls = torch.empty(A, device="cuda")
        ctx.ppo_loss_gaussian(dev(head.detach().numpy()), dev(log_std.detach().numpy().reshape(-1)), dev(values.detach().numpy()),
                              dev(act), dev(old_lp), dev(adv), dev(ret), hyper, losses, dhead, dls, dval, ws)
        assert nerr(dls.cpu().numpy(), log_std.grad.numpy().reshape(-1)) <= 1e-4
    else:
        ctx.ppo_loss_discrete(dev(head.detach().numpy()), dev(values.detach().numpy()), dev(act, torch.int32), dev(old_lp),
                              dev(adv), dev(ret), hyper, losses, dhead, dval, ws)
    np.testing.assert_allclose(losses.cpu().numpy(), [float(lp), float(lv), float(ent), float(total)], rtol=1e-4, atol=1e-6)
    assert nerr(dhead.cpu().numpy(), head.grad.numpy()) <= 1e-4
    assert nerr(dval.cpu().numpy(), values.grad.numpy()) <= 1e-5


# ---------------------------------------------------------------- rollout pieces --------------
def test_gather_rows(ctx):
    rng = np.random.default_rng(0)
    src = rng.standard_normal((1000, 7)).astype(np.float32)
    idx = rng.permutation(1000)[:300].astype(np.int32)
    out = ctx.gather_rows(dev(src), dev(idx, torch.int32))
    np.testing.assert_array_equal(out.cpu().numpy(), src[idx])          # bit-exact


def test_store_step_casts_and_layout(ctx):
    for cont in (False, True):
        N_, D, A, T = 37, 5, 3, 4
        rng = np.random.default_rng(1)
        obs = torch.zeros(T, N_, D, device="cuda"); nobs = torch.zeros(T, N_, D, device="cuda")
        actions = torch.zeros((T, N_, A) if cont else (T, N_), dtype=torch.float32 if cont else torch.int32, device="cuda")
        rew = torch.zeros(T, N_, device="cuda"); te = torch.zeros(T, N_, device="cuda"); tr = torch.zeros(T, N_, device="cuda")
        nbytes = ctx.step_record_bytes(N_, D, A, cont)
        for t in range(T):
            o = rng.standard_normal((N_, D)).astype(np.float32); no = rng.standard_normal((N_, D)).astype(np.float32)
            r = rng.standard_normal(N_); term = rng.random(N_) < 0.3; trunc = rng.random(N_) < 0.3
            a = rng.standard_normal((N_, A)).astype(np.float32) if cont else rng.integers(0, A, N_).astype(np.int64)
            rec = o.tobytes() + no.tobytes() + r.astype(np.float64).tobytes() + a.tobytes() + term.astype(np.uint8).tobytes() + trunc.astype(np.uint8).tobytes()
            assert len(rec) == nbytes
            drec = torch.frombuffer(bytearray(rec + b"\0" * (-len(rec) % 8)), dtype=torch.uint8).cuda()
            ctx.buffer_store_step(drec, t, N_, D, A, cont, obs, nobs, actions, rew, te, tr)
            np.testing.assert_array_equal(obs[t].cpu().numpy(), o)
            np.testing.assert_array_equal(nobs[t].cpu().numpy(), no)
            np.testing.assert_array_equal(rew[t].cpu().numpy(), r.astype(np.float32))
            np.testing.assert_array_equal(te[t].cpu().numpy(), term.astype(np.float32))      # masks bit-exact
            np.testing.assert_array_equal(tr[t].cpu().numpy(), trunc.astype(np.float32))
            np.testing.assert_array_equal(actions[t].cpu().numpy(), a.astype(np.float32 if cont else np.int32))


def test_sample_categorical_distribution_and_determinism(ctx):
    N_, A = 200000, 4
    logits = torch.tensor([[0.1, -1.0, 2.0, 0.5]], device="cuda").repeat(N_, 1).contiguous()
    lp = torch.empty(N_, device="cuda")
    a1 = ctx.sample_categorical(logits, seed=42, counter=7, log_probs=lp)
    a2 = ctx.sample_categorical(logits, seed=42, counter=7)
    assert torch.equal(a1, a2)                                           # deterministic under its own seed
    a3 = ctx.sample_categorical(logits[1000:3000].contiguous(), seed=42, counter=7, env_offset=1000)
    assert torch.equal(a1[1000:3000], a3)                                # keyed by global env id, not launch shape
    a4 = ctx.sample_categorical(logits, seed=42, counter=8)
    assert not torch.equal(a1, a4)
    p = torch.softmax(logits[0], -1).cpu().numpy()
    counts = np.bincount(a1.cpu().numpy(), minlength=A)
    chi2 = ((counts - N_ * p) ** 2 / (N_ * p)).sum()
    assert chi2 < 25.0, (chi2, counts)                                   # 3 dof, p ~ 1e-5
    ref_lp = torch.log_softmax(logits[0], -1)[a1]
    np.testing.assert_allclose(lp.cpu().numpy(), ref_lp.cpu().numpy(), rtol=1e-5, atol=1e-6)


def test_sample_gaussian_distribution(ctx):
    N_, A = 200000, 3
    mean = torch.tensor([[0.5, -2.0, 1.0]], device="cuda").repeat(N_, 1).contiguous()
    log_std = torch.tensor([0.0, -1.0, 0.7], device="cuda")
    lp = torch.empty(N_, device="cuda")
    a = ctx.sample_gaussian(mean, log_std, seed=1, counter=3, log_probs=lp)
    x = a.cpu().numpy()
    np.testing.assert_allclose(x.mean(0), [0.5, -2.0, 1.0], atol=0.02)
    np.testing.assert_allclose(x.std(0), np.exp([0.0, -1.0, 0.7]), rtol=0.02)
    assert abs(np.corrcoef(x[:, 0], x[:, 1])[0, 1]) < 0.01
    ref = torch.distributions.Normal(mean, log_std.exp()).log_prob(a).sum(-1)
    np.testing.assert_allclose(lp.cpu().numpy(), ref.cpu().numpy(), rtol=1e-4, atol=1e-4)


def test_gae_back_to_back_launches_with_settled_inputs(ctx):
    """Programmatic dependent launch: consecutive launches overlap (inputs requested before griddepcontrol.wait); results
    must not change, including when consecutive launches write the same output buffers."""
    T, N = 128, 4096
    rng = np.random.default_rng(5)
    sets = []
    for k in range(6):
        r = rng.standard_normal((T, N)).astype(np.float32)
        te = (rng.random((T, N)) < 0.01).astype(np.float32)
        tr = ((rng.random((T, N)) < 0.01) & (te == 0)).astype(np.float32)
        v = rng.standard_normal((T, N)).astype(np.float32)
        nv = rng.standard_normal((T, N)).astype(np.float32)
        sets.append((r, te, tr, v, nv))
    dsets = [[dev(x) for x in s_] for s_ in sets]
    outs = [(torch.empty(T, N, device="cuda"), torch.empty(T, N, device="cuda")) for _ in sets]
    shared_adv, shared_ret = torch.empty(T, N, device="cuda"), torch.empty(T, N, device="cuda")
    torch.cuda.synchronize()
    for rep in range(3):
        for k, d_ in enumerate(dsets):
            ctx.gae(*d_, 0.99, 0.95, advantages=outs[k][0], returns=outs[k][1], inputs_settled=True)
    for k, d_ in enumerate(dsets):                       # same outputs every launch: the last writer must win
        ctx.gae(*d_, 0.99, 0.95, advantages=shared_adv, returns=shared_ret, inputs_settled=True)
    torch.cuda.synchronize()
    for k, s_ in enumerate(sets):
        ref, ref_r = CO.gae(*s_, 0.99, 0.95)
        assert nerr(outs[k][0].cpu().numpy(), ref) <= 1e-5
        assert nerr(outs[k][1].cpu().numpy(), ref_r) <= 1e-5
    ref, ref_r = CO.gae(*sets[-1], 0.99, 0.95)
    assert nerr(shared_adv.cpu().numpy(), ref) <= 1e-5
    assert nerr(shared_ret.cpu().numpy(), ref_r) <= 1e-5


# ---------------------------------------------------------------- tensor-core (3xTF32 tcgen05) path ----
@pytest.mark.parametrize("D,H,A,rows", [(64, 256, 4, 4096), (64, 256, 4, 5000), (32, 128, 3, 2048), (16, 512, 5, 1024)])
def test_tensor_core_forward_matches_fp32_path_and_oracle(ctx, D, H, A, rows):
    from diamond.flat import FlatMlp
    rng = np.random.default_rng(H + rows)
    p = rand_params(rng, O.DISCRETE_PARAM_NAMES, D, H, A, False)
    fm = FlatMlp(D, H, A, False)
    flat = fm.pack(p, device="cuda")
    obs = rng.standard_normal((rows, D)).astype(np.float32)
    ref_out, ref_v = O.mlp_forward(p, torch.as_tensor(obs), False)
    ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, rows, False) // 4 + 512, device="cuda")
    res = {}
    for tc in (1, 0):
        ctx.set_option("tensor_cores", tc)
        out = torch.empty(rows, A, device="cuda"); val = torch.empty(rows, device="cuda")
        ctx.mlp_forward(fm.desc, flat, dev(obs), rows, 3, out, val, ws)
        torch.cuda.synchronize()
        res[tc] = (out.cpu().numpy(), val.cpu().numpy())
    ctx.set_option("tensor_cores", 1)
    for tc in (1, 0):
        assert nerr(res[tc][0], ref_out.numpy()) <= 1e-5, tc
        assert nerr(res[tc][1], ref_v.numpy()) <= 1e-5, tc
    assert nerr(res[1][0], res[0][0]) <= 1e-5
    assert nerr(res[1][1], res[0][1]) <= 1e-5


def test_tensor_core_training_step_matches_fp32_path(ctx):
    from diamond import _native as N
    from diamond.flat import FlatMlp
    D, H, A, B, M = 64, 256, 4, 8192, 4096
    rng = np.random.default_rng(11)
    p = rand_params(rng, O.DISCRETE_PARAM_NAMES, D, H, A, False)
    fm = FlatMlp(D, H, A, False)
    flat = fm.pack(p, device="cuda")
    obs = dev(rng.standard_normal((B, D)).astype(np.float32)); act = dev(rng.integers(0, A, B), torch.int32)
    old_lp = dev((rng.standard_normal(B) * 0.3 - 1.0).astype(np.float32))
    adv = dev(rng.standard_normal(B).astype(np.float32)); ret = dev(rng.standard_normal(B).astype(np.float32))
    idx = dev(rng.permutation(B)[:M].astype(np.int32), torch.int32)
    hyper, cfg = make_hyper(N, M)
    ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, M, True) // 4 + 512, device="cuda")
    out = {}
    for tc in (1, 0):
        ctx.set_option("tensor_cores", tc)
        grads = torch.zeros(fm.total, device="cuda"); losses = torch.zeros(4, device="cuda")
        ctx.mlp_grad_minibatch(fm.desc, flat, grads, obs, act, old_lp, adv, ret, None, idx, M, hyper, losses, ws)
        torch.cuda.synchronize()
        out[tc] = (grads.cpu().numpy(), losses.cpu().numpy())
    ctx.set_option("tensor_cores", 1)
    gv0 = fm.views(torch.as_tensor(out[0][0]))
    for tc in (1,):
        np.testing.assert_allclose(out[tc][1], out[0][1], rtol=1e-5, atol=1e-7)
        gv = fm.views(torch.as_tensor(out[tc][0]))
        for n in O.DISCRETE_PARAM_NAMES:
            assert nerr(gv[n].numpy(), gv0[n].numpy()) <= 2e-5, (tc, n)


@pytest.mark.parametrize("M", [4096, 5000, 19200])
def test_row_sweep_and_l2_hint_options_do_not_change_the_update(ctx, M):
    """row_sweep (gemm_tc3.cu dppo_tc3_gemm): alternating sweep directions of consecutive launches, cacheable d3 stores and the L2
    evict-first hints only move cache lines -- bit-identical gradients; the reversed head kernel (bit 1) and the reversed dgrad launch
    (column sums of the bias gradient) re-order fp32 partial sums -- equal to 2e-5.  Forward outputs are bit-identical throughout.
    Ragged M covers the half-width tail tiles and the clipped last row tile in both directions."""
    from diamond import _native as N
    from diamond.flat import FlatMlp
    D, H, A = 64, 256, 4
    B = 2 * M
    rng = np.random.default_rng(M)
    p = rand_params(rng, O.DISCRETE_PARAM_NAMES, D, H, A, False)
    fm = FlatMlp(D, H, A, False)
    flat = fm.pack(p, device="cuda")
    obs = dev(rng.standard_normal((B, D)).astype(np.float32)); act = dev(rng.integers(0, A, B), torch.int32)
    old_lp = dev((rng.standard_normal(B) * 0.3 - 1.0).astype(np.float32))
    adv = dev(rng.standard_normal(B).astype(np.float32)); ret = dev(rng.standard_normal(B).astype(np.float32))
    idx = dev(rng.permutation(B)[:M].astype(np.int32), torch.int32)
    hyper, cfg = make_hyper(N, M)
    ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, M, True) // 4 + 512, device="cuda")
    wsf = torch.empty(ctx.mlp_workspace_bytes(fm.desc, B, False) // 4 + 512, device="cuda")
    out = {}
    try:
        for sweep in (0, 1, 2, 4 | 8 | 16, 31):
            ctx.set_option("row_sweep", sweep)
            grads = torch.zeros(fm.total, device="cuda"); losses = torch.zeros(4, device="cuda")
            ctx.mlp_grad_minibatch(fm.desc, flat, grads, obs, act, old_lp, adv, ret, None, idx, M, hyper, losses, ws)
            logits = torch.empty(B, A, device="cuda"); val = torch.empty(B, device="cuda")
            ctx.mlp_forward(fm.desc, flat, obs, B, 3, logits, val, wsf)
            torch.cuda.synchronize()
            out[sweep] = (grads.cpu().numpy(), losses.cpu().numpy(), logits.cpu().numpy(), val.cpu().numpy())
    finally:
        ctx.set_option("row_sweep", 31)
    for sweep in (1, 2, 28, 31):
        assert np.array_equal(out[sweep][2], out[0][2]) and np.array_equal(out[sweep][3], out[0][3]), sweep
    assert np.array_equal(out[28][0], out[0][0]) and np.array_equal(out[28][1], out[0][1])
    gv0 = fm.views(torch.as_tensor(out[0][0]))
    for sweep in (1, 2, 31):
        np.testing.assert_allclose(out[sweep][1], out[0][1], rtol=1e-5, atol=1e-7)
        gv = fm.views(torch.as_tensor(out[sweep][0]))
        for n in O.DISCRETE_PARAM_NAMES:
            assert nerr(gv[n].numpy(), gv0[n].numpy()) <= 2e-5, (sweep, n)


# fp32 parity needs ~1e-6; single-pass TF32 would sit near 5e-4 on these products
TC_TOL = 3e-5


@pytest.mark.parametrize("M,N,K", [(4096, 256, 64), (4096, 256, 256), (4096, 512, 256), (5000, 256, 512), (1024, 128, 64),
                                   (65536, 256, 256)])
def test_tc_linear_forward_vs_fp64(ctx, M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    C, _ = ctx.tc_linear(1, A, W, False, bias=b)
    ref = torch.tanh(A.double() @ W.double().T + b.double())
    assert (C.double() - ref).abs().max().item() <= TC_TOL


@pytest.mark.parametrize("M,N,K", [(4096, 256, 512), (4096, 256, 256), (5000, 256, 256), (65536, 256, 512)])
def test_tc_linear_dgrad_vs_fp64(ctx, M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M + N + K + 1)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(K, N, device="cuda", generator=g) / K ** 0.5
    Hact = torch.tanh(torch.randn(M, N, device="cuda", generator=g))
    C, cs = ctx.tc_linear(2, A, W, True, Hact=Hact, colsum=True)
    ref = (A.double() @ W.double()) * (1.0 - Hact.double() ** 2)
    assert (C.double() - ref).abs().max().item() <= TC_TOL * max(1.0, ref.abs().max().item())
    col = ref.sum(0)
    cs = cs[:cs.shape[0] // 5]                          # per-CTA partial rows; the rest are per-quadrant working rows
    assert (cs.double().sum(0) - col).abs().max().item() <= 3e-5 * max(1.0, col.abs().max().item())


@pytest.mark.parametrize("M,N1,N2", [(4096, 256, 256), (4096, 512, 256), (4096, 256, 64), (5000, 256, 256), (65536, 512, 256),
                                     (65536, 256, 64), (4100, 128, 128)])
def test_tc_wgrad_vs_fp64(ctx, M, N1, N2):
    g = torch.Generator(device="cuda").manual_seed(M + N1 + N2)
    Dm = torch.randn(M, N1, device="cuda", generator=g)
    Hm = torch.randn(M, N2, device="cuda", generator=g)
    dW = ctx.tc_wgrad(Dm, Hm)
    ref = Dm.double().T @ Hm.double()
    assert ((dW.double() - ref).abs().max() / ref.abs().max()).item() <= TC_TOL
    # bit-reproducible (fixed summation order)
    assert torch.equal(dW, ctx.tc_wgrad(Dm, Hm))


# ---------------------------------------------------------------- device permutation + shard filter ----
@pytest.mark.parametrize("n", [1, 2, 5, 1000, 4096, 65537, 524288])
def test_permutation_device_is_a_keyed_permutation(ctx, n):
    """Fast-mode generator (SURVEY 2.2 K4a): a bijection of [0, n) for every (seed, counter), deterministic, key-sensitive."""
    out = torch.empty(n, dtype=torch.int32, device="cuda")
    a = ctx.permutation_device(7, 0, n, out).cpu().numpy().copy()
    assert np.array_equal(np.sort(a), np.arange(n))
    assert np.array_equal(a, ctx.permutation_device(7, 0, n, out).cpu().numpy())              # pure function of (seed, counter)
    if n >= 1000:
        b = ctx.permutation_device(7, 1, n, out).cpu().numpy().copy()
        c = ctx.permutation_device(8, 0, n, out).cpu().numpy().copy()
        assert np.array_equal(np.sort(b), np.arange(n)) and np.array_equal(np.sort(c), np.arange(n))
        for other in (b, c):
            assert (a == other).mean() < max(0.01, 10.0 / n)                                                 # different keys: unrelated permutations
        assert (a == np.arange(n)).mean() < max(0.01, 10.0 / n)                                              # few fixed points
        # positions look uniform: the first tenth of the outputs covers all ten value deciles evenly (chi^2, 9 dof, p ~ 1e-6 at 45)
        head = a[:n // 10]
        obs_counts = np.bincount((head.astype(np.int64) * 10 // n).clip(0, 9), minlength=10)
        chi2 = ((obs_counts - head.size / 10) ** 2 / (head.size / 10)).sum()
        assert chi2 < 45, chi2
        # neighbours are not kept together: correlation of consecutive outputs is ~ 0
        assert abs(np.corrcoef(a[:-1], a[1:])[0, 1]) < max(0.02, 5.0 / np.sqrt(n))


@pytest.mark.parametrize("T,NL,world,MB", [(8, 6, 2, 4), (32, 40, 4, 8), (128, 512, 8, 8), (16, 3, 3, 2)])
def test_perm_shard_filter_matches_oracle(ctx, T, NL, world, MB):
    from diamond.agents import permutation_plan
    from oracle.dp_oracle import shard_filter
    NG, B = NL * world, T * NL * world
    if B % MB:
        pytest.skip("shape does not divide")
    rng = np.random.default_rng(T + NL)
    perm = rng.permutation(B).astype(np.int32)
    rows = permutation_plan(T * NL, world, MB, True)["rows"]
    for rank in range(world):
        idx = torch.full((MB * rows,), 12345, dtype=torch.int32, device="cuda")
        counts = torch.zeros(MB, dtype=torch.int32, device="cuda"); over = torch.zeros(1, dtype=torch.int32, device="cuda")
        ctx.perm_shard_filter(dev(perm, torch.int32), B, NG, rank * NL, NL, MB, rows, idx, counts, over)
        ref_idx, ref_counts, ref_over = shard_filter(perm, NG, rank * NL, NL, MB, rows)
        assert np.array_equal(idx.cpu().numpy().reshape(MB, rows), ref_idx)                    # bit-exact, order preserved, -1 padding
        assert np.array_equal(counts.cpu().numpy(), ref_counts) and int(over) == ref_over == 0
    # too small a pad: surplus dropped, flag raised (the caller treats it as an error)
    tiny = max(1, (B // MB) // world // 2)
    idx = torch.empty(MB * tiny, dtype=torch.int32, device="cuda")
    counts = torch.zeros(MB, dtype=torch.int32, device="cuda"); over = torch.zeros(1, dtype=torch.int32, device="cuda")
    ctx.perm_shard_filter(dev(perm, torch.int32), B, NG, 0, NL, MB, tiny, idx, counts, over)
    ref_idx, ref_counts, ref_over = shard_filter(perm, NG, 0, NL, MB, tiny)
    assert int(over) == ref_over == 1 and np.array_equal(idx.cpu().numpy().reshape(MB, tiny), ref_idx)


@pytest.mark.parametrize("D,H,A,cont,B,M,pad", [(8, 64, 4, False, 600, 200, 56), (64, 256, 4, False, 8192, 3000, 1096),
                                                (5, 64, 3, True, 512, 100, 28), (32, 128, 3, False, 4096, 2000, 48),
                                                (64, 256, 2, True, 4096, 1501, 35)])
def test_padding_rows_contribute_nothing(ctx, D, H, A, cont, B, M, pad):
    """idx < 0 marks a padding row (fixed-shape steps under data parallelism): losses and the flat gradient of M real rows
    followed by `pad` padding rows equal those of the M rows alone (same loss denominator)."""
    from diamond import _native as N
    from diamond.flat import FlatMlp
    rng = np.random.default_rng(B + M)
    names = O.CONTINUOUS_PARAM_NAMES if cont else O.DISCRETE_PARAM_NAMES
    p = rand_params(rng, names, D, H, A, cont)
    fm = FlatMlp(D, H, A, cont)
    flat = fm.pack(p, device="cuda")
    obs = dev(rng.standard_normal((B, D)).astype(np.float32))
    act = dev(rng.standard_normal((B, A)).astype(np.float32)) if cont else dev(rng.integers(0, A, B), torch.int32)
    old_lp = dev((rng.standard_normal(B) * 0.3 - 1.0).astype(np.float32))
    adv = dev(rng.standard_normal(B).astype(np.float32)); ret = dev(rng.standard_normal(B).astype(np.float32))
    real = rng.permutation(B)[:M].astype(np.int32)
    # padding interleaved and at the end
    padded = np.concatenate([real[:M // 2], np.full(pad // 2, -1, np.int32), real[M // 2:], np.full(pad - pad // 2, -1, np.int32)])
    hyper, _ = make_hyper(N, M)
    outs = []
    for idx in (real, padded):
        rows = idx.size
        ws = torch.empty(ctx.mlp_workspace_bytes(fm.desc, rows, True) // 4 + 512, device="cuda")
        grads = torch.full((fm.total,), 7.0, device="cuda"); losses = torch.zeros(4, device="cuda")
        ctx.mlp_grad_minibatch(fm.desc, flat, grads, obs, act, old_lp, adv, ret, None, dev(idx, torch.int32), rows, hyper, losses, ws)
        torch.cuda.synchronize()
        outs.append((grads.cpu().numpy(), losses.cpu().numpy()))
    np.testing.assert_allclose(outs[1][1], outs[0][1], rtol=2e-6, atol=1e-7)
    gv0, gv1 = fm.views(torch.as_tensor(outs[0][0])), fm.views(torch.as_tensor(outs[1][0]))
    for n in names:
        assert nerr(gv1[n].numpy(), gv0[n].numpy()) <= 5e-6, n
