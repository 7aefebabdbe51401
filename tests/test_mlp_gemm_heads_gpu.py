"""GEMM heads of the default MLP networks (dppo_mlp_grad_minibatch_gemm_heads, csrc/heads.cu wide_loss_kernel / critic_value_kernel):
hidden widths up to 2048 and up to 1024 actions, through the C ABI and PPO / ContinuousPPO, against the float64 oracle
(oracle/ppo_oracle.py).

The mirror below restates the host-side condition of the fused head kernel (heads.cu head_train_supported): the shapes
dppo_mlp_grad_minibatch takes.  FusedMlpEngine runs every other shape on GEMM heads."""
import numpy as np
import pytest
import torch

from oracle import ppo_oracle as O

gpu = pytest.mark.gpu


# ---------------------------------------------------------------- mirror of heads.cu head_train_supported --------------------
def fused_heads_supported(H, A):
    """1 <= A <= 32, H <= 512, and Wa | wc plus eight per-warp [(A+1), H] accumulators (at least the flush scratch) in 200 KB."""
    if not (1 <= A <= 32 and 1 <= H <= 512):
        return False
    acc = max(8 * (A + 1) * H, 8 * (2 * H + 100))
    return ((A + 1) * H + acc) * 4 <= 200 * 1024


GEMM_MAX_HIDDEN, GEMM_MAX_ACT = 2048, 1024

# (H, A, continuous, fused?, why)
SHAPE_TABLE = [
    (64, 4, False, True, "default width"),
    (64, 1, False, True, "A = 1"),
    (37, 1, True, True, "odd H, A = 1, Gaussian"),
    (150, 32, False, True, "A = 32, H not a multiple of 4"),
    (512, 10, True, True, "largest A at H = 512"),
    (256, 21, False, True, "largest A at H = 256"),
    (384, 13, True, True, "largest A at H = 384"),
    (512, 11, False, False, "shared-memory band"),
    (512, 12, False, False, "shared-memory band (the shape dppo_mlp_grad_minibatch refuses)"),
    (512, 17, True, False, "shared-memory band, Gaussian (Humanoid-shaped)"),
    (256, 22, False, False, "shared-memory band"),
    (384, 14, True, False, "shared-memory band"),
    (513, 1, False, False, "H > 512"),
    (1024, 4, False, False, "H > 512"),
    (64, 33, True, False, "A > 32"),
    (256, 100, False, False, "A > 32"),
    (1024, 64, False, False, "H > 512 and A > 32"),
    (2048, 1024, False, False, "the GEMM-head bound"),
    (2047, 1023, True, False, "odd H and A just under the bound"),
]


def test_fused_heads_condition_mirror_and_case_table():
    """CPU: the Python mirror, the case table and dppo_mlp_fused_heads_supported agree; the table covers every reason the fused
    kernel refuses (H > 512, A > 32, the shared-memory band, both at once), odd H, A = 1, both distributions and the bound."""
    import ctypes
    from diamond import _native as N
    ws = lambda H, A, cont: N.load_library().dppo_mlp_gemm_heads_workspace_bytes(ctypes.byref(N.MlpDesc(8, H, A, int(cont))),
                                                                                 ctypes.c_int64(256))
    for H, A, cont, fused, why in SHAPE_TABLE:
        assert fused_heads_supported(H, A) == fused, (H, A, why)
        assert N.fused_heads_supported(N.MlpDesc(8, H, A, int(cont))) == fused, (H, A, why)
        assert ws(H, A, cont) > 0
    rows = [(H, A) for H, A, *_ in SHAPE_TABLE]
    assert any(H > 512 and A <= 32 for H, A in rows) and any(A > 32 and H <= 512 for H, A in rows)
    assert any(H > 512 and A > 32 for H, A in rows)
    band = [(H, A) for H, A in rows if H <= 512 and A <= 32 and not fused_heads_supported(H, A)]
    assert (512, 12) in band and {H for H, _ in band} >= {256, 384, 512}
    assert any(H % 4 for H, _ in rows) and any(A == 1 for _, A in rows) and (GEMM_MAX_HIDDEN, GEMM_MAX_ACT) in rows
    assert {r[2] for r in SHAPE_TABLE} == {False, True}
    # the band boundaries of the issue's table: (A + 1) H > 5688
    for H in (256, 384, 512):
        first = min(A for A in range(1, 33) if not fused_heads_supported(H, A))
        assert (first + 1) * H > 5688 and first * H <= 5688, H
    # above the bound: no workspace, and the fused kernel does not take it either
    for H, A in ((GEMM_MAX_HIDDEN + 1, 4), (64, GEMM_MAX_ACT + 1)):
        assert ws(H, A, False) == 0
        assert not fused_heads_supported(H, A)


# ---------------------------------------------------------------- helpers -----------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as N
    return N.get_context(0)


def dev(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x)).to(device="cuda", dtype=dtype).contiguous()


def nerr(a, ref):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(a - ref).max() / max(np.abs(ref).max(), 1e-30)


def rand_params(rng, D, H, A, cont, scale=0.3):
    head = "actor_mean_head" if cont else "actor_head"
    shapes = {"base.0.weight": (H, D), "base.0.bias": (H,), "base.2.weight": (H, H), "base.2.bias": (H,),
              f"{head}.0.weight": (H, H), f"{head}.0.bias": (H,), f"{head}.2.weight": (A, H), f"{head}.2.bias": (A,),
              "critic_head.0.weight": (H, H), "critic_head.0.bias": (H,), "critic_head.2.weight": (1, H),
              "critic_head.2.bias": (1,), "actor_log_std": (1, A)}
    names = O.CONTINUOUS_PARAM_NAMES if cont else O.DISCRETE_PARAM_NAMES
    p = {}
    for n in names:
        s = scale if len(shapes[n]) == 1 else 1.0 / np.sqrt(shapes[n][-1])
        p[n] = torch.as_tensor((rng.standard_normal(shapes[n]) * s).astype(np.float32))
    return names, p


def make_hyper(M, den=None, adv_norm=False, adv_count=0):
    from diamond import _native as N
    cfg = O.default_cfg()
    h = N.Hyper()
    h.ppo_clip, h.value_loss_weight, h.entropy_beta = cfg["ppo_clip"], cfg["value_loss_weight"], cfg["entropy_beta"]
    h.grad_norm_clip, h.adam_eps, h.lr = cfg["grad_norm_clip"], cfg["adam_eps"], cfg["lr"]
    h.beta1, h.beta2, h.step = 0.9, 0.999, 1
    h.advantage_norm, h.adv_count, h.loss_denominator = int(adv_norm), adv_count, M if den is None else den
    return h, cfg


class Problem:
    """Random network + rollout of B samples.  Old log-probs are the float64 log-probs plus N(0, 0.1) noise, so the ratios
    straddle the clip range without sitting on its edges."""

    def __init__(self, D, H, A, cont, B, seed):
        from diamond.flat import FlatMlp
        rng = np.random.default_rng(seed)
        self.D, self.H, self.A, self.cont, self.B = D, H, A, cont, B
        self.names, self.p = rand_params(rng, D, H, A, cont)
        self.p64 = {k: v.double() for k, v in self.p.items()}
        self.fm = FlatMlp(D, H, A, cont)
        self.flat = self.fm.pack(self.p, device="cuda")
        self.obs = rng.standard_normal((B, D)).astype(np.float32)
        self.act = rng.standard_normal((B, A)).astype(np.float32) if cont else rng.integers(0, A, B)
        out, _ = O.mlp_forward(self.p64, torch.as_tensor(self.obs).double(), cont)
        t_act = torch.as_tensor(self.act)
        lp = (O.normal_log_prob(out, self.p64["actor_log_std"].expand_as(out), t_act.double()) if cont
              else O.categorical_log_prob(out, t_act)[0])
        self.old_lp = (lp.numpy() + rng.standard_normal(B) * 0.1).astype(np.float32)
        self.adv = (rng.standard_normal(B) * 2 + 0.5).astype(np.float32)
        self.ret = rng.standard_normal(B).astype(np.float32)
        self.d = dict(obs=dev(self.obs), act=dev(self.act, torch.float32 if cont else torch.int32), old_lp=dev(self.old_lp),
                      adv=dev(self.adv), ret=dev(self.ret))
        a64 = self.adv.astype(np.float64)
        self.stats = torch.tensor([a64.sum(), (a64 ** 2).sum(), 0.0, 0.0], dtype=torch.float64, device="cuda")

    def reference(self, rows, den, adv_norm):
        """float64 losses and gradients of the rows `rows` with loss denominator den."""
        a = self.adv.astype(np.float64)
        if adv_norm:
            mu = a.sum() / self.B
            var = max(((a ** 2).sum() - a.sum() * mu) / (self.B - 1), 0.0)
            a = (a - mu) / (np.sqrt(var) + 1e-6)
        sel = torch.as_tensor(np.asarray(rows, dtype=np.int64))
        t = lambda x: torch.as_tensor(x).double() if x.dtype.kind == "f" else torch.as_tensor(x)
        _, cfg = make_hyper(1)
        losses, g = O.loss_and_grads(self.p64, t(self.obs)[sel], t(self.act)[sel], t(self.old_lp)[sel], torch.as_tensor(a)[sel],
                                     t(self.ret)[sel], cfg, self.cont)
        k = len(rows) / den                                       # the oracle divides by its row count
        return {n: v * k for n, v in losses.items()}, {n: v * k for n, v in g.items()}

    def run(self, ctx, idx, M, den, adv_norm, gemm=True, grads=None):
        hyper, _ = make_hyper(M, den, adv_norm, self.B)
        grads = torch.full((self.fm.total,), 7.0, device="cuda") if grads is None else grads
        losses = torch.zeros(4, device="cuda")
        sumsq = torch.zeros(ctx.grad_sumsq_bytes(self.fm.total) // 8 + 1, dtype=torch.float64, device="cuda")
        hyper.grad_sumsq = sumsq.data_ptr()
        nb = ctx.mlp_gemm_heads_workspace_bytes(self.fm.desc, M) if gemm else ctx.mlp_workspace_bytes(self.fm.desc, M, True)
        ws = torch.empty(nb // 4 + 64, device="cuda")
        fn = ctx.mlp_grad_minibatch_gemm_heads if gemm else ctx.mlp_grad_minibatch
        d = self.d
        fn(self.fm.desc, self.flat, grads, d["obs"], d["act"], d["old_lp"], d["adv"], d["ret"], self.stats if adv_norm else None,
           None if idx is None else dev(idx, torch.int32), M, hyper, losses, ws)
        torch.cuda.synchronize()
        return grads, losses, sumsq


def check_against(pb, grads, losses, sumsq, ref_losses, ref_g, M=0):
    # the MLP tests' 2e-5 per tensor; 5e-5 where the trunk runs on the 3xTF32 tensor cores at H >= 512 (rows >= 1024, H a multiple of
    # 256; measured 3.1e-5 at H = 1024 and 2.3e-5 at H = 512 with D = 376).  Losses: rtol 1e-5, with an absolute floor of 1e-5 of the
    # largest loss (the policy term is a mean of terms of both signs and can cancel)
    tol = 5e-5 if (M >= 1024 and pb.H >= 512 and pb.H % 256 == 0) else 2e-5
    ref_l = np.array([ref_losses[k] for k in ("policy", "value", "entropy", "total")])
    np.testing.assert_allclose(losses.cpu().numpy(), ref_l, rtol=1e-5, atol=1e-5 * np.abs(ref_l).max())
    gv = pb.fm.views(grads)
    for n in pb.names:
        e = nerr(gv[n].cpu().numpy(), ref_g[n].numpy())
        assert e <= tol, (n, e)
    used = torch.zeros(pb.fm.total, dtype=torch.bool)
    for n, (off, shape) in pb.fm.slices.items():
        used[off:off + int(np.prod(shape))] = True
    assert float(grads.cpu()[~used].abs().sum()) == 0.0                 # padding between tensors is zero
    ref_sq = sum(float((ref_g[n] ** 2).sum()) for n in pb.names)
    got_sq = float(sumsq[:-1].sum())
    assert abs(got_sq - ref_sq) <= 1e-4 * ref_sq, (got_sq, ref_sq)     # the clip norm dppo_clip_adam_step reads


# One row per case: shapes the fused kernel refuses for each reason, odd widths, both distributions, the bound.
# opts: "norm" (advantage normalisation), "den2" (loss denominator 2 M).  M >= 1024 runs the trunk on the tensor cores.
CASES = [
    # id              D    H     A     cont   B     M     opts
    ("h1024-a4",     24, 1024,    4, False, 2048, 1024, "norm"),
    ("h512-a17-g",  376,  512,   17, True,  2048, 1100, ""),
    ("h256-a100",   128,  256,  100, False, 3000, 1500, "den2"),
    ("h512-a12",      8,  512,   12, False,  600,  256, "norm den2"),
    ("h150-a33-g",   10,  150,   33, True,   700,  333, "den2"),
    ("h37-a1",        5,   37,    1, False,  400,  131, "norm"),
    ("h600-a3-g",    12,  600,    3, True,  1500, 1100, ""),
    ("h2048-a1024",  16, 2048, 1024, False,  300,  200, ""),
]
CASE_IDS = [c[0] for c in CASES]


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_gemm_heads_grad_minibatch_vs_fp64(ctx, case):
    """Every gradient tensor (2e-5 of its largest entry), the four losses (rtol 1e-5), zero padding between tensors and the
    grad_sumsq partials against float64, with idx NULL (rows 0..M-1) and with a permutation slice."""
    cid, D, H, A, cont, B, M, opts = case
    pb = Problem(D, H, A, cont, B, seed=H * 7 + A)
    den = 2 * M if "den2" in opts else M
    norm = "norm" in opts
    perm = np.random.default_rng(A).permutation(B)[:M].astype(np.int32)
    for idx in (None, perm):
        rows = np.arange(M) if idx is None else perm
        ref_losses, ref_g = pb.reference(rows, den, norm)
        check_against(pb, *pb.run(ctx, idx, M, den, norm), ref_losses, ref_g, M)


@gpu
@pytest.mark.parametrize("D,H,A,cont,B,M", [(16, 256, 100, False, 4096, 1500), (12, 1024, 5, True, 1024, 700)])
def test_gemm_heads_padding_rows_and_reproducibility(ctx, D, H, A, cont, B, M):
    """Padding rows (idx < 0, interleaved and at the end) contribute nothing: losses and gradient equal those of the real rows
    alone; a repeated call is bit-identical."""
    pb = Problem(D, H, A, cont, B, seed=M)
    rng = np.random.default_rng(1)
    real = rng.permutation(B)[:M].astype(np.int32)
    pad = 77
    padded = np.concatenate([real[:M // 2], np.full(pad // 2, -1, np.int32), real[M // 2:], np.full(pad - pad // 2, -1, np.int32)])
    g0, l0, _ = pb.run(ctx, real, M, M, True)
    g1, l1, _ = pb.run(ctx, padded, padded.size, M, True)
    g2, l2, _ = pb.run(ctx, padded, padded.size, M, True)
    assert torch.equal(g1, g2) and torch.equal(l1, l2)
    np.testing.assert_allclose(l1.cpu().numpy(), l0.cpu().numpy(), rtol=2e-6, atol=1e-7)
    gv0, gv1 = pb.fm.views(g0), pb.fm.views(g1)
    for n in pb.names:
        assert nerr(gv1[n].cpu().numpy(), gv0[n].cpu().numpy()) <= 5e-6, n
    ref_losses, ref_g = pb.reference(real, M, True)
    check_against(pb, g1, l1, pb.run(ctx, padded, padded.size, M, True)[2], ref_losses, ref_g)


@gpu
@pytest.mark.parametrize("D,H,A,cont,B,M", [(64, 256, 4, False, 4096, 1500), (17, 96, 7, False, 700, 333), (64, 256, 6, True, 4096, 1500),
                                            (10, 150, 32, False, 1000, 333), (6, 512, 9, True, 2048, 700), (8, 64, 2, True, 512, 128)])
def test_gemm_heads_match_fused_heads(ctx, D, H, A, cont, B, M):
    """On shapes the fused head kernel also runs, the two entries agree per tensor to 5e-5 of its largest entry (two fp32 results that
    differ in summation order only; the few-entry actor_log_std gradient of a 2-dim Gaussian differs by 4.2e-5)."""
    pb = Problem(D, H, A, cont, B, seed=D + H + A)
    idx = np.random.default_rng(2).permutation(B)[:M].astype(np.int32)
    gf, lf, sf = pb.run(ctx, idx, M, M, True, gemm=False)
    gg, lg, sg = pb.run(ctx, idx, M, M, True, gemm=True)
    np.testing.assert_allclose(lg.cpu().numpy(), lf.cpu().numpy(), rtol=1e-5, atol=1e-5 * float(lf.abs().max()))
    gvf, gvg = pb.fm.views(gf), pb.fm.views(gg)
    for n in pb.names:
        assert nerr(gvg[n].cpu().numpy(), gvf[n].cpu().numpy()) <= 5e-5, n
    assert abs(float(sg[:-1].sum()) - float(sf[:-1].sum())) <= 1e-5 * float(sf[:-1].sum())


@gpu
def test_gemm_heads_refuse_above_the_bound(ctx):
    from diamond import _native as N
    for H, A in ((GEMM_MAX_HIDDEN + 1, 4), (64, GEMM_MAX_ACT + 1)):
        pb_desc = N.MlpDesc(4, H, A, 0)
        from diamond.flat import FlatMlp
        fm = FlatMlp(4, H, A, False)
        P = torch.zeros(fm.total, device="cuda")
        hyper, _ = make_hyper(8)
        z = torch.zeros(8, device="cuda")
        ws = torch.empty(1024, device="cuda")
        with pytest.raises(N.NativeError, match=str(GEMM_MAX_HIDDEN if H > GEMM_MAX_HIDDEN else GEMM_MAX_ACT)):
            ctx.mlp_grad_minibatch_gemm_heads(pb_desc, P, torch.zeros_like(P), torch.zeros(8, 4, device="cuda"),
                                              torch.zeros(8, dtype=torch.int32, device="cuda"), z, z, z, None, None, 8, hyper,
                                              torch.zeros(4, device="cuda"), ws)
    # the context keeps working
    pb = Problem(5, 37, 1, False, 64, seed=3)
    ref_losses, ref_g = pb.reference(np.arange(64), 64, False)
    check_against(pb, *pb.run(ctx, None, 64, 64, False), ref_losses, ref_g)


# ---------------------------------------------------------------- forward -----------------------------------------------------
@gpu
@pytest.mark.parametrize("D,H,A,cont,B", [(24, 1024, 4, False, 3000), (376, 512, 17, True, 2000), (128, 256, 100, False, 1500),
                                          (16, 2048, 1024, False, 300), (10, 150, 33, True, 700), (12, 600, 3, True, 1100)])
def test_gemm_heads_forward_and_next_values_vs_fp64(ctx, D, H, A, cont, B):
    """dppo_mlp_forward with heads 1, 2, 3 (rows chunked, and gathered through idx) and dppo_mlp_next_values at shapes past the
    fused head evaluation, against float64 (1e-5 of the largest entry)."""
    pb = Problem(D, H, A, cont, B, seed=B)
    ref_out, ref_v = O.mlp_forward(pb.p64, torch.as_tensor(pb.obs).double(), cont)
    ref_out, ref_v = ref_out.numpy(), ref_v.numpy()
    ws = torch.empty(ctx.mlp_workspace_bytes(pb.fm.desc, B // 2 + 3, False) // 4, device="cuda")       # two chunks
    obs = pb.d["obs"]
    for heads in (1, 2, 3):
        out = torch.full((B, A), 9.0, device="cuda") if heads & 1 else None
        val = torch.full((B,), 9.0, device="cuda") if heads & 2 else None
        ctx.mlp_forward(pb.fm.desc, pb.flat, obs, B, heads, out, val, ws)
        torch.cuda.synchronize()
        if heads & 1:
            assert nerr(out.cpu().numpy(), ref_out) <= 1e-5, heads
        if heads & 2:
            assert nerr(val.cpu().numpy(), ref_v) <= 1e-5, heads
    idx = np.random.default_rng(0).permutation(B)[:B // 3].astype(np.int32)
    out = torch.empty(idx.size, A, device="cuda"); val = torch.empty(idx.size, device="cuda")
    ctx.mlp_forward(pb.fm.desc, pb.flat, obs, idx.size, 3, out, val, ws, idx=dev(idx, torch.int32))
    torch.cuda.synchronize()
    assert nerr(out.cpu().numpy(), ref_out[idx]) <= 1e-5 and nerr(val.cpu().numpy(), ref_v[idx]) <= 1e-5
    # next_values: values[t + 1] where the environment went on, V(next_obs) on finished steps and the last row
    N_ = 50
    T = B // N_
    rng = np.random.default_rng(4)
    nobs = rng.standard_normal((T * N_, D)).astype(np.float32)
    term = (rng.random((T, N_)) < 0.1).astype(np.float32)
    trunc = ((rng.random((T, N_)) < 0.05) & (term == 0)).astype(np.float32)
    values = rng.standard_normal((T, N_)).astype(np.float32)
    nv = torch.full((T, N_), 9.0, device="cuda")
    nws = torch.empty(ctx.mlp_next_values_workspace_bytes(pb.fm.desc, T, N_), dtype=torch.uint8, device="cuda")
    ctx.mlp_next_values(pb.fm.desc, pb.flat, dev(nobs), dev(term), dev(trunc), dev(values), nv, nws)
    torch.cuda.synchronize()
    got = nv.cpu().numpy()
    _, v_next = O.mlp_forward(pb.p64, torch.as_tensor(nobs).double(), cont)
    v_next = v_next.numpy().reshape(T, N_)
    need = (term != 0) | (trunc != 0)
    need[-1] = True
    assert np.array_equal(got[:-1][~need[:-1]], values[1:][~need[:-1]])
    assert np.abs(got[need] - v_next[need]).max() <= 1e-5 * max(1.0, np.abs(v_next).max())


# ---------------------------------------------------------------- standalone loss (custom network_cls) --------------------------
def torch_loss(head, values, log_std, act, old_lp, adv, ret, cont, M, cfg):
    if cont:
        dist = torch.distributions.Normal(head, log_std.exp().expand_as(head))
        new_lp, ent = dist.log_prob(act).sum(-1), dist.entropy().sum(-1).sum() / M
    else:
        dist = torch.distributions.Categorical(logits=head)
        new_lp, ent = dist.log_prob(act), dist.entropy().sum() / M
    ratio = (new_lp - old_lp).exp()
    eps = cfg["ppo_clip"]
    lp = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - eps, 1 + eps)).sum() / M
    lv = 0.5 * ((values - ret) ** 2).sum() / M
    return lp, lv, ent, lp + cfg["value_loss_weight"] * lv - cfg["entropy_beta"] * ent


@gpu
@pytest.mark.parametrize("A,cont,row_std", [(100, False, False), (1024, False, False), (40, True, False), (77, True, True)])
def test_standalone_loss_above_32_actions_vs_fp64(ctx, A, cont, row_std):
    """dppo_ppo_loss_* at A > 32 (lanes stride over the actions) against torch autograd in float64: losses, d/dhead, d/dvalues and
    d/dlog_std (shared [A] vector or per row)."""
    M = 1000
    rng = np.random.default_rng(A)
    head = torch.as_tensor(rng.standard_normal((M, A))).requires_grad_(True)
    values = torch.as_tensor(rng.standard_normal(M)).requires_grad_(True)
    log_std = torch.as_tensor(rng.standard_normal((M if row_std else 1, A)) * 0.2).requires_grad_(True)
    act = torch.as_tensor(rng.standard_normal((M, A))) if cont else torch.as_tensor(rng.integers(0, A, M))
    with torch.no_grad():
        lp_ref = (torch.distributions.Normal(head, log_std.exp().expand_as(head)).log_prob(act).sum(-1) if cont
                  else torch.distributions.Categorical(logits=head).log_prob(act))
    old_lp = lp_ref + torch.as_tensor(rng.standard_normal(M) * 0.1)
    adv, ret = torch.as_tensor(rng.standard_normal(M)), torch.as_tensor(rng.standard_normal(M))
    hyper, cfg = make_hyper(M)
    ref = torch_loss(head, values, log_std, act, old_lp, adv, ret, cont, M, cfg)
    ref[3].backward()
    f = lambda x: dev(x.detach().numpy())
    ws = torch.empty(ctx.ppo_loss_workspace_bytes(M, A) // 4 + 16, device="cuda")
    losses = torch.zeros(4, device="cuda"); dhead = torch.empty(M, A, device="cuda"); dval = torch.empty(M, device="cuda")
    if cont:
        dls = torch.empty((M, A) if row_std else (A,), device="cuda")
        ls_in = f(log_std) if row_std else f(log_std.reshape(-1))
        ctx.ppo_loss_gaussian(f(head), ls_in, f(values), f(act), f(old_lp), f(adv), f(ret), hyper, losses, dhead, dls, dval, ws,
                              log_std_row_stride=A if row_std else 0)
        torch.cuda.synchronize()
        assert nerr(dls.cpu().numpy().reshape(-1), log_std.grad.numpy().reshape(-1)) <= 2e-5
    else:
        ctx.ppo_loss_discrete(f(head), f(values), dev(act.numpy(), torch.int32), f(old_lp), f(adv), f(ret), hyper, losses, dhead, dval, ws)
        torch.cuda.synchronize()
    np.testing.assert_allclose(losses.cpu().numpy(), [float(x) for x in ref], rtol=1e-5, atol=1e-7)
    assert nerr(dhead.cpu().numpy(), head.grad.numpy()) <= 2e-5
    assert nerr(dval.cpu().numpy(), values.grad.numpy()) <= 1e-5


@gpu
def test_sample_categorical_100_actions(ctx):
    """Categorical sampling at A = 100 (the rollout of a 100-action PPO): chi^2 against softmax(logits), deterministic per seed."""
    N_, A = 400000, 100
    g = torch.Generator().manual_seed(0)
    row = torch.randn(A, generator=g) * 1.5
    logits = row.cuda().repeat(N_, 1).contiguous()
    lp = torch.empty(N_, device="cuda")
    a1 = ctx.sample_categorical(logits, seed=9, counter=3, log_probs=lp)
    assert torch.equal(a1, ctx.sample_categorical(logits, seed=9, counter=3))
    p = torch.softmax(row.double(), -1).numpy()
    counts = np.bincount(a1.cpu().numpy(), minlength=A)
    big = N_ * p >= 5                                                    # pool cells with fewer than 5 expected draws
    obs_c, exp_c = counts[big].astype(np.float64), N_ * p[big]
    if (~big).any():
        obs_c, exp_c = np.append(obs_c, counts[~big].sum()), np.append(exp_c, N_ * p[~big].sum())
    chi2 = ((obs_c - exp_c) ** 2 / exp_c).sum()
    dof = obs_c.size - 1
    assert chi2 < dof + 6 * np.sqrt(2 * dof), (chi2, dof)               # ~ p 1e-5
    np.testing.assert_allclose(lp.cpu().numpy(), torch.log_softmax(row, -1)[a1.cpu()].numpy(), rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------- agent level ---------------------------------------------------
@gpu
@pytest.mark.parametrize("kind,D,A,H,N_,T", [("ppo", 8, 4, 1024, 16, 64), ("ppo", 12, 100, 256, 32, 48), ("cont", 376, 17, 512, 16, 64)])
def test_agent_gemm_heads_match_autograd_engine(kind, D, A, H, N_, T):
    """PPO at H = 1024, PPO with 100 actions and a Humanoid-shaped ContinuousPPO (D = 376, A = 17, H = 512) run the fused engine on
    GEMM heads; after one learn() (1 epoch x 2 minibatches) the parameters equal the same network run under torch autograd
    (AutogradEngine) on the same rollout to 1e-4 of each tensor's largest entry, floored at 1e-2: the biases start at zero, so after
    two Adam steps they are O(lr) and their relative error measures Adam's g / sqrt(v) amplification of fp32 rounding in gradients
    near eps, not the gradient.  Losses to 1e-4."""
    from diamond import PPO, PPOConfig, ContinuousPPO, ContinuousPPOConfig, envs
    from diamond.agents import FusedMlpEngine, AutogradEngine, RolloutBuffer
    from diamond.networks import ActorCriticNetwork, ContinuousActorCriticNetwork
    cont = kind == "cont"
    Agent, Cfg, Net = (ContinuousPPO, ContinuousPPOConfig, ContinuousActorCriticNetwork) if cont else (PPO, PPOConfig, ActorCriticNetwork)

    class Same(Net):
        pass

    agents = []
    for cls in (Net, Same):
        cfg = Cfg(num_envs=N_, rollout_steps=T, num_epochs=1, num_minibatches=2, verbose=False, network_hidden_dim=H, seed=3,
                  total_steps=N_ * T * 100)
        agents.append(Agent(lambda: envs.SyntheticEnv(D, A, continuous=cont), cfg, network_cls=cls))
    fused, auto = agents
    assert isinstance(fused.engine, FusedMlpEngine) and isinstance(auto.engine, AutogradEngine)
    assert not fused.engine.fused_heads
    auto.network.load_state_dict(fused.network.state_dict())
    rng = np.random.default_rng(H + A)
    exp = [[rng.standard_normal((N_, D)).astype(np.float32), rng.standard_normal((N_, D)).astype(np.float32),
            rng.standard_normal((N_, A)).astype(np.float32) if cont else rng.integers(0, A, N_), rng.standard_normal(N_),
            rng.random(N_) < 0.05, np.zeros(N_, bool)] for _ in range(T)]
    for ag in (fused, auto):
        buf = RolloutBuffer.from_lists(ag.ctx, exp, cont, ag.device)
        np.random.seed(8)
        ag.learn(buf)
    torch.cuda.synchronize()
    for (k, p), (_, q) in zip(fused.network.named_parameters(), auto.network.named_parameters()):
        err = float((p - q).abs().max() / q.abs().max().clamp_min(1e-2))
        assert err <= 1e-4, (k, err)
    assert float((fused.engine.last_losses - auto.engine.last_losses).abs().max()) <= 1e-4


@gpu
def test_device_rollout_graph_replay_with_100_actions():
    """Device-resident synthetic environments, 100 actions at H = 256 (forward GEMM heads + sampling): the CUDA-graph replay of a
    rollout records exactly what the eager launches record, and the recorded values / log-probs are what the float64 module
    computes from the recorded observations."""
    from diamond import PPO, PPOConfig
    from diamond.envs import DeviceVectorEnv
    N_, T, H, A, D = 64, 16, 256, 100, 12
    recs = []
    for use_graphs in (True, False):
        cfg = PPOConfig(num_envs=N_, rollout_steps=T, verbose=False, seed=6, total_steps=N_ * T * 100, network_hidden_dim=H)
        agent = PPO(DeviceVectorEnv.factory("Synthetic", seed=6, obs_dim=D, n_actions=A), cfg)
        agent.engine.use_graphs = use_graphs
        agent.ticker = None
        agent.current_observations, _ = agent.envs.reset(seed=6)
        out = []
        for _ in range(4):
            ro = agent.rollout()
            out.append([getattr(ro, k).clone() for k in ("obs", "actions", "rewards", "terminations", "truncations", "logp", "values")])
        torch.cuda.synchronize()
        if use_graphs:
            assert agent._rollout_graph is not None, "graph path was not taken"
            net64 = agent.network.double().cpu()
        recs.append(out)
    for a, b in zip(*recs):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    for obs, actions, *_, logp, values in recs[0]:
        with torch.inference_mode():
            logits, v = net64.get_logits_and_values(obs.double().cpu().reshape(T * N_, D))
        lp = torch.distributions.Categorical(logits=logits).log_prob(actions.cpu().reshape(-1).long())
        assert float((v.reshape(-1) - values.cpu().double().reshape(-1)).abs().max()) <= 1e-5
        assert float((lp - logp.cpu().double().reshape(-1)).abs().max()) <= 1e-5


# ---------------------------------------------------------------- up to 32 actions: unchanged ------------------------------------
# (A, continuous) cases of the standalone loss that stay on loss_rows_kernel; tests/golden/loss_le32.npz holds what the library
# computed before the GEMM-head path existed (B200).
LE32_CASES = [(5, False), (32, False), (7, True), (32, True)]


def le32_inputs(A, cont):
    M = 1000
    rng = np.random.default_rng(100 + A + 50 * cont)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    act = f(M, A) if cont else rng.integers(0, A, M).astype(np.int32)
    return dict(M=M, head=f(M, A), values=f(M), log_std=f(A) * 0.2, act=act, old_lp=f(M) * 0.3 - (1.5 * A if cont else 1.5),
                adv=f(M), ret=f(M))


def run_le32(ctx, A, cont):
    x = le32_inputs(A, cont)
    M = x["M"]
    hyper, _ = make_hyper(M)
    ws = torch.empty(ctx.ppo_loss_workspace_bytes(M, A) // 4 + 16, device="cuda")
    losses = torch.zeros(4, device="cuda"); dhead = torch.empty(M, A, device="cuda"); dval = torch.empty(M, device="cuda")
    dls = torch.zeros(A, device="cuda")
    if cont:
        ctx.ppo_loss_gaussian(dev(x["head"]), dev(x["log_std"]), dev(x["values"]), dev(x["act"]), dev(x["old_lp"]), dev(x["adv"]),
                              dev(x["ret"]), hyper, losses, dhead, dls, dval, ws)
    else:
        ctx.ppo_loss_discrete(dev(x["head"]), dev(x["values"]), dev(x["act"], torch.int32), dev(x["old_lp"]), dev(x["adv"]),
                              dev(x["ret"]), hyper, losses, dhead, dval, ws)
    torch.cuda.synchronize()
    return dict(losses=losses.cpu().numpy(), dhead=dhead.cpu().numpy(), dval=dval.cpu().numpy(), dls=dls.cpu().numpy())


@gpu
def test_standalone_loss_up_to_32_actions_is_unchanged(ctx):
    """A <= 32 keeps loss_rows_kernel: losses and gradients are bit-identical to those recorded before the wide path existed."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "loss_le32.npz"))
    for A, cont in LE32_CASES:
        out = run_le32(ctx, A, cont)
        for k, v in out.items():
            assert np.array_equal(v, g[f"A{A}_c{int(cont)}.{k}"]), (A, cont, k)
