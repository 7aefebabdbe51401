"""The one-launch update of the default 64-wide networks (dppo_small_update, csrc/small_net.cu, DESIGN.md §4b) against float64.

dppo_small_update runs every optimiser step of a learn() inside one thread-block cluster: gather, forward, loss, backward, the
gradient reduce-scatter over distributed shared memory, clip, Adam and the parameter all-gather.  Its launch plan (small_plan) picks
the cluster size CL and the tile height RT from the minibatch rows.  Each CTA then loops over ceil(rows per CTA / RT) tiles and
accumulates its gradient partial across them.  The mirror below restates small_plan, the row bound and
dppo_small_update_supported, so that the case table can name, and a CPU test can check, the plan class of every case.

The reference is torch autograd in float64 on oracle.ppo_oracle.mlp_forward.  Its loss is written out with an explicit live-row
mask and loss denominator, so padding rows and the denominator are checked against the math, not against a second copy of the
kernel's hand-derived gradient.  Clip and Adam follow in float64 (oracle.ppo_oracle.adam_step_).  The gradient is compared tensor by
tensor: Adam's update m / (sqrt(v) + eps) hardly moves when one tensor's gradient is off by a constant factor."""
import math

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as O

gpu = pytest.mark.gpu

LR, ADAM_EPS, BETA1, BETA2 = 3e-4, 1e-5, 0.9, 0.999
ADAM_T0 = 5                                                 # Adam step of the first update: moments are non-zero, bias corrections matter


# ---------------------------------------------------------------- mirror of csrc/small_net.cu --------------------------------
HN, AMAX, ROWS_MAX = 64, 8, 128                             # hidden width, actions, minibatch rows per CTA
SMEM_BUDGET = 220 * 1024                                    # dynamic shared memory dppo_small_update_supported allows


def layout_total(D, H, A, cont):
    """dppo_mlp_layout_compute: floats in the flat buffer, every tensor padded to 4 floats."""
    up = lambda n: (n + 3) // 4 * 4
    return (up(H * D) + up(H) + up(H * H) + up(H) + up(2 * H * H) + up(2 * H) + up(A * H) + up(A) + up(H) + up(1)
            + (up(A) if cont else 0))


def small_smem_bytes(total, D, RT, CL):
    """small_smem_bytes: parameters + gradient partial, three Adam slices, the activation tiles, head outputs and scratch."""
    RS = RT + 4
    SL = ((total + CL - 1) // CL + 3) & ~3
    fl = 2 * total + 3 * SL + (D + 4 * HN + 2 * 2 * HN) * RS + RT * AMAX + RT + (2 * AMAX + 1) * RS + 8
    return fl * 4 + 64


def small_supported(D, H, A, cont):
    """dppo_small_update_supported.  The shared-memory budget (taken at RT = 32, CL = 8, the largest plan) bounds obs_dim well below
    64: 30 at 8 actions, 36 at 1."""
    if not (H == HN and 1 <= D <= 64 and 1 <= A <= AMAX):
        return False
    total = layout_total(D, H, A, cont)
    return total % 4 == 0 and small_smem_bytes(total, D, 32, 8) <= SMEM_BUDGET


def small_plan(rows):
    """small_plan: (RT, CL)."""
    CL = 16 if rows > 8 * 32 else 8
    RT = 16 if (rows + CL - 1) // CL <= 16 else 32
    return RT, CL


def rows_accepted(rows):
    """dppo_small_update's row bound: 1 <= rows <= CL * ROWS_MAX (2048)."""
    RT, CL = small_plan(rows)
    return 1 <= rows <= CL * ROWS_MAX


def plan_class(rows):
    """What one CTA of the launch sees: (CL, RT, tiles per CTA), rows of every CTA, whether a CTA's last tile is ragged and whether
    every tile of every CTA is full."""
    RT, CL = small_plan(rows)
    per = (rows + CL - 1) // CL
    counts = []
    for rank in range(CL):
        lo = min(rows, rank * per)
        counts.append(min(rows, lo + per) - lo)
    tiles = (per + RT - 1) // RT
    return dict(CL=CL, RT=RT, tiles=tiles, counts=counts, zero_ctas=sum(c == 0 for c in counts),
                ragged=any(c % RT for c in counts if c), full=all(c == tiles * RT for c in counts))


def max_supported_obs(A, cont):
    return max(D for D in range(1, 65) if small_supported(D, HN, A, cont))


# One row per case: the plan class it is meant to run, then the shapes.  opts: "pad" padding rows (idx < 0, scattered and a padded
# tail), "norm" advantage normalisation from fp64 statistics, "den2" loss denominator 2 * rows (what data parallelism passes).
# D = 30 with 8 actions and D = 36 with 1 action are the largest obs_dim the shared-memory budget admits.
CASES = [
    # id          D   A  cont   rows   opts            (CL, RT, tiles)
    ("r1",        3,  2, False,    1, "norm",          (8, 16, 1)),
    ("r9-g",      5,  3, True,     9, "",              (8, 16, 1)),
    ("r100-pad",  1,  4, False,  100, "pad den2",      (8, 16, 1)),
    ("r200",     17,  8, False,  200, "",              (8, 32, 1)),
    ("r256-g",    7,  2, True,   256, "norm",          (8, 32, 1)),
    ("r300-g",   30,  8, True,   300, "den2",          (16, 32, 1)),
    ("r512-g",   36,  1, True,   512, "norm",          (16, 32, 1)),
    ("r700-pad", 11,  5, False,  700, "pad norm",      (16, 32, 2)),
    ("r1000-g",   8,  6, True,  1000, "den2",          (16, 32, 2)),
    ("r1024",     4,  2, False, 1024, "norm",          (16, 32, 2)),
    ("r1300",    24,  8, False, 1300, "",              (16, 32, 3)),
    ("r1800-g",  30,  8, True,  1800, "pad",           (16, 32, 4)),
    ("r2048",     3,  3, False, 2048, "norm den2",     (16, 32, 4)),
]
CASE_IDS = [c[0] for c in CASES]

# Several optimiser steps in one launch: a 4-tile case, a 2-tile Gaussian case with a ragged tile, and one with fewer rows than CTAs.
MULTI_CASES = [
    # id            D   A  cont   rows  steps  opts
    ("r2048-s2",    5,  4, False, 2048,  2,    "norm"),
    ("r740-g-s3",   9,  3, True,   740,  3,    "pad norm den2"),
    ("r5-s8",       4,  2, False,    5,  8,    "pad norm"),
]
MULTI_IDS = [c[0] for c in MULTI_CASES]


def test_small_net_plan_mirror_and_case_table():
    """CPU: the mirror of the layout and of the shape rule agree with the library; the case table names each case's plan class and
    covers every class: CL 8 with RT 16 and 32, CL 16 with 1 to 4 tiles, a ragged last tile, all tiles full, CTAs without rows,
    both distributions, A = 1 and 8, D = 1, an odd D and the largest supported D, padding, advantage normalisation on and off, and a
    loss denominator of 2 * rows."""
    import ctypes
    from diamond import _native as N
    lib = N.load_library()
    for cont in (False, True):
        for A in (1, 2, 5, 8, 9):
            for D in (1, 2, 7, 29, 30, 31, 33, 36, 37, 64, 65):
                for H in (63, 64, 65):
                    desc = N.MlpDesc(D, H, A, int(cont))
                    assert layout_total(D, H, A, cont) == N.mlp_layout(desc).total, (D, H, A, cont)
                    assert small_supported(D, H, A, cont) == bool(lib.dppo_small_update_supported(ctypes.byref(desc))), (D, H, A, cont)
    assert max_supported_obs(8, False) == max_supported_obs(8, True) == 30
    assert max_supported_obs(1, False) == max_supported_obs(1, True) == 36
    assert not small_supported(64, HN, 1, False)                    # obs_dim 64 is over the shared-memory budget at every A
    # row bound and plan classes over every accepted row count
    assert [rows_accepted(r) for r in (0, 1, 2048, 2049)] == [False, True, True, False]
    seen = set()
    for rows in range(1, 2049):
        c = plan_class(rows)
        assert max(c["counts"]) <= ROWS_MAX and sum(c["counts"]) == rows
        seen.add((c["CL"], c["RT"], c["tiles"]))
    assert seen == {(8, 16, 1), (8, 32, 1), (16, 32, 1), (16, 32, 2), (16, 32, 3), (16, 32, 4)}
    # the table
    classes = set()
    for cid, D, A, cont, rows, opts, want in CASES:
        c = plan_class(rows)
        assert (c["CL"], c["RT"], c["tiles"]) == want, cid
        assert small_supported(D, HN, A, cont), cid
        classes.add(want)
    assert classes == seen
    pc = {cid: plan_class(rows) for cid, _, _, _, rows, _, _ in CASES}
    assert pc["r1000-g"]["ragged"] and pc["r1000-g"]["counts"][0] == 63 and pc["r1000-g"]["counts"][-1] == 55
    assert pc["r1024"]["full"] and pc["r2048"]["full"] and pc["r1024"]["tiles"] == 2 and pc["r2048"]["tiles"] == 4
    assert pc["r1"]["zero_ctas"] == 7 and pc["r9-g"]["zero_ctas"] == 3
    assert {c[3] for c in CASES} == {False, True}
    assert {1, 8} <= {c[2] for c in CASES}
    Ds = {c[1] for c in CASES}
    assert 1 in Ds and any(D % 2 for D in Ds if D > 1)
    assert any(D == max_supported_obs(A, cont) for _, D, A, cont, *_ in CASES if A == 8)
    assert any(D == max_supported_obs(A, cont) for _, D, A, cont, *_ in CASES if A == 1)
    opts = [c[5].split() for c in CASES]
    assert any("pad" in o for o in opts) and any("den2" in o for o in opts)
    assert any("norm" in o for o in opts) and any("norm" not in o for o in opts)
    assert any(c[6][2] >= 2 and "pad" in c[5].split() for c in CASES)
    # the multi-step cases: 4 tiles, a ragged 2-tile Gaussian case, fewer rows than CTAs; S in {2, 3, 8}
    m = {cid: plan_class(rows) for cid, _, _, _, rows, _, _ in MULTI_CASES}
    assert m["r2048-s2"]["tiles"] == 4 and m["r740-g-s3"]["tiles"] == 2 and m["r740-g-s3"]["ragged"] and m["r5-s8"]["zero_ctas"] == 3
    assert sorted(c[5] for c in MULTI_CASES) == [2, 3, 8]
    assert all(small_supported(D, HN, A, cont) for _, D, A, cont, *_ in MULTI_CASES)


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


def make_hyper(rows, den, norm, adv_count, max_norm):
    from diamond import _native as N
    cfg = O.default_cfg(grad_norm_clip=max_norm)
    h = N.Hyper()
    h.ppo_clip, h.value_loss_weight, h.entropy_beta = cfg["ppo_clip"], cfg["value_loss_weight"], cfg["entropy_beta"]
    h.grad_norm_clip, h.adam_eps, h.lr = max_norm, ADAM_EPS, LR
    h.beta1, h.beta2, h.step = BETA1, BETA2, ADAM_T0
    h.advantage_norm, h.adv_count, h.loss_denominator = int(norm), adv_count, den
    return h, cfg


def step_consts(t0, steps):
    """[steps][2] = {sqrt(1 - beta2^t), -lr / (1 - beta1^t)} computed in double, as the agents do."""
    c = np.array([[math.sqrt(1.0 - BETA2 ** t), -(LR / (1.0 - BETA1 ** t))] for t in range(t0, t0 + steps)], dtype=np.float32)
    return c


class Problem:
    """Random 64-wide network, a buffer of B samples and an Adam state of an earlier step.

    The old log-probs are the float64 log-probs of the initial parameters minus log(r), so each row's first ratio is r: drawn from
    [0.55, 0.75], [0.85, 1.15] or [1.25, 1.6].  Rows fall on both sides of both clip edges and no ratio sits near one."""

    def __init__(self, D, A, cont, B, seed):
        from diamond.flat import FlatMlp
        rng = np.random.default_rng(seed)
        self.D, self.A, self.cont, self.B = D, A, cont, B
        self.fm = FlatMlp(D, HN, A, cont)
        self.names = O.CONTINUOUS_PARAM_NAMES if cont else O.DISCRETE_PARAM_NAMES
        shapes = {n: s for n, (_, s) in self.fm.slices.items()}
        self.p32 = {}
        for n in self.names:
            s = shapes[n]
            scale = 0.3 if (len(s) == 1 or n == "actor_log_std") else 1.0 / np.sqrt(s[-1])
            self.p32[n] = torch.as_tensor((rng.standard_normal(s) * scale).astype(np.float32))
        self.p64 = {n: v.double() for n, v in self.p32.items()}
        self.obs = rng.standard_normal((B, D)).astype(np.float32)
        self.act = rng.standard_normal((B, A)).astype(np.float32) if cont else rng.integers(0, A, B).astype(np.int32)
        lp = self.log_probs(self.p64).numpy()
        band = rng.choice(3, B, p=[0.25, 0.5, 0.25])
        lo, hi = np.array([0.55, 0.85, 1.25])[band], np.array([0.75, 1.15, 1.6])[band]
        r = lo + (hi - lo) * rng.random(B)
        self.old_lp = (lp - np.log(r)).astype(np.float32)
        self.adv = (rng.standard_normal(B) * 2 + 0.5).astype(np.float32)
        self.ret = rng.standard_normal(B).astype(np.float32)
        self.M0 = self.fm.pack({n: rng.standard_normal(shapes[n]) * 1e-2 for n in self.names})
        self.V0 = self.fm.pack({n: rng.uniform(1e-4, 4e-4, shapes[n]) for n in self.names})
        self.P0 = self.fm.pack(self.p32)
        self._d = None

    def log_probs(self, p):
        out, _ = O.mlp_forward(p, torch.as_tensor(self.obs).double(), self.cont)
        if self.cont:
            return O.normal_log_prob(out, p["actor_log_std"].expand_as(out), torch.as_tensor(self.act).double())
        return O.categorical_log_prob(out, torch.as_tensor(self.act))[0]

    def adv_used(self, norm):
        a = self.adv.astype(np.float64)
        if norm:                                                          # ppo.py:243 from fp64 sums, unbiased
            mu = a.sum() / self.B
            var = max(((a ** 2).sum() - a.sum() * mu) / (self.B - 1), 0.0)
            a = (a - mu) / (np.sqrt(var) + 1e-6)
        return torch.as_tensor(a)

    def step_indices(self, rows, steps, pad, seed):
        """steps distinct slices of one permutation of the buffer; with pad, every odd step (every step when steps == 1) gets ~10 %
        scattered padding rows and a padded tail, keeping row 0 live."""
        rng = np.random.default_rng(seed)
        idx = rng.permutation(self.B)[:rows * steps].reshape(steps, rows).astype(np.int32)
        if pad:
            for k in range(steps):
                if steps > 1 and k % 2 == 0:
                    continue
                m = rng.random(rows) < 0.1
                m[-max(1, rows // 16):] = True
                m[0] = False
                idx[k][m] = -1
        return idx.reshape(-1)

    def device(self):
        if self._d is None:
            a64 = self.adv.astype(np.float64)
            self._d = dict(obs=dev(self.obs), act=dev(self.act, torch.float32 if self.cont else torch.int32), old_lp=dev(self.old_lp),
                           adv=dev(self.adv), ret=dev(self.ret),
                           stats=torch.tensor([a64.sum(), (a64 ** 2).sum(), 0.0, 0.0], dtype=torch.float64, device="cuda"))
        return self._d

    # ---- float64 reference ---------------------------------------------------------------------------------------------
    def reference_grad(self, p64, idx, den, norm, cfg):
        """Losses (policy, value, entropy, total) and the gradient of one step, by torch autograd in float64.  Padding rows
        (idx < 0) are gathered from row 0 and masked out of every loss term."""
        p = {n: v.detach().clone().requires_grad_(True) for n, v in p64.items()}
        idx = torch.as_tensor(np.asarray(idx, dtype=np.int64))
        live = (idx >= 0).double()
        src = idx.clamp(min=0)
        out, v = O.mlp_forward(p, torch.as_tensor(self.obs).double()[src], self.cont)
        if self.cont:
            log_std = p["actor_log_std"].expand_as(out)
            new_lp = O.normal_log_prob(out, log_std, torch.as_tensor(self.act).double()[src])
            ent = (0.5 + 0.5 * math.log(2 * math.pi) + log_std).sum(-1)
        else:
            lsm = torch.log_softmax(out, -1)
            new_lp = lsm.gather(-1, torch.as_tensor(self.act).long()[src].unsqueeze(-1)).squeeze(-1)
            ent = -(lsm.exp() * lsm).sum(-1)
        ratio = torch.exp(new_lp - torch.as_tensor(self.old_lp).double()[src])
        adv = self.adv_used(norm)[src]
        eps = cfg["ppo_clip"]
        pol = (live * torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - eps, 1 + eps))).sum() / den
        val = 0.5 * (live * (v - torch.as_tensor(self.ret).double()[src]) ** 2).sum() / den
        entropy = (live * ent).sum() / den
        total = pol + cfg["value_loss_weight"] * val - cfg["entropy_beta"] * entropy
        total.backward()
        r = ratio.detach()[live.bool()]
        margin = float(torch.minimum((r - (1 - eps)).abs(), (r - (1 + eps)).abs()).min())
        assert margin > 1e-3, f"a live ratio is {margin:.2e} from a clip edge: change the case's seed"
        return np.array([float(x.detach()) for x in (pol, val, entropy, total)]), {n: p[n].grad for n in self.names}

    def reference_update(self, p64, M64, V64, idx, rows, steps, den, norm, max_norm):
        """steps sequential float64 optimiser steps: gradient -> clip_grad_norm_ -> Adam.  Returns per-step losses, the last step's
        pre-clip norm and clipped gradient, and the final parameters and moments."""
        _, cfg = make_hyper(rows, den, norm, self.B, max_norm)
        p = {n: v.clone() for n, v in p64.items()}
        state = dict(step=ADAM_T0 - 1, exp_avg={n: v.clone() for n, v in M64.items()}, exp_avg_sq={n: v.clone() for n, v in V64.items()})
        losses = []
        for k in range(steps):
            l, g = self.reference_grad(p, idx[k * rows:(k + 1) * rows], den, norm, cfg)
            losses.append(l)
            norm64 = O.clip_grad_norm_(g, self.names, max_norm)
            O.adam_step_(p, g, state, self.names, LR, ADAM_EPS, BETA1, BETA2)
        return dict(losses=np.array(losses), norm=norm64, grads=g, P=p, M=state["exp_avg"], V=state["exp_avg_sq"])

    # ---- the kernel ------------------------------------------------------------------------------------------------------
    def run(self, ctx, idx, rows, steps, den, norm, max_norm, P=None, M=None, V=None, t0=ADAM_T0):
        """One dppo_small_update launch of `steps` steps on P / M / V (copies of the initial state unless given; updated in place)."""
        d = self.device()
        P = self.P0.cuda() if P is None else P
        M = self.M0.cuda() if M is None else M
        V = self.V0.cuda() if V is None else V
        hyper, _ = make_hyper(rows, den, norm, self.B, max_norm)
        G = torch.full((self.fm.total,), 7.0, device="cuda")
        losses = torch.full((steps, 4), 7.0, device="cuda")
        gn = torch.full((1,), 7.0, device="cuda")
        ctx.small_update(self.fm.desc, P, G, M, V, d["obs"], d["act"], d["old_lp"], d["adv"], d["ret"], d["stats"] if norm else None,
                         dev(idx, torch.int32), rows, steps, hyper, dev(step_consts(t0, steps)), losses, gn)
        torch.cuda.synchronize()
        return dict(P=P, M=M, V=V, G=G, losses=losses, gn=gn)

    def named64(self, flat):
        return {n: v.detach().cpu().double() for n, v in self.fm.views(flat.detach().cpu()).items()}

    def padding_mask(self):
        used = torch.zeros(self.fm.total, dtype=torch.bool)
        for off, shape in self.fm.slices.values():
            used[off:off + int(np.prod(shape))] = True
        return ~used


def case_setup(D, A, cont, rows, opts, steps, seed):
    opts = opts.split()
    B = max(rows * steps + rows // 2 + 7, 16)
    pb = Problem(D, A, cont, B, seed)
    idx = pb.step_indices(rows, steps, "pad" in opts, seed + 1)
    return pb, idx, (2 * rows if "den2" in opts else rows), "norm" in opts


def test_fp64_reference_matches_oracle_loss_and_grads():
    """CPU: without padding and with denominator = rows, the autograd reference equals the oracle's hand-derived loss_and_grads."""
    for D, A, cont in ((5, 3, False), (4, 2, True)):
        pb = Problem(D, A, cont, 300, seed=D)
        rows = 200
        idx = np.random.default_rng(0).permutation(pb.B)[:rows]
        for norm in (False, True):
            _, cfg = make_hyper(rows, rows, norm, pb.B, 0.5)
            losses, g = pb.reference_grad(pb.p64, idx, rows, norm, cfg)
            t = torch.as_tensor(idx.astype(np.int64))
            ol, og = O.loss_and_grads(pb.p64, torch.as_tensor(pb.obs).double()[t],
                                      torch.as_tensor(pb.act).double()[t] if cont else torch.as_tensor(pb.act)[t],
                                      torch.as_tensor(pb.old_lp).double()[t], pb.adv_used(norm)[t], torch.as_tensor(pb.ret).double()[t],
                                      cfg, cont)
            np.testing.assert_allclose(losses, [ol[k] for k in ("policy", "value", "entropy", "total")], rtol=1e-12, atol=1e-14)
            for n in pb.names:
                assert nerr(g[n].numpy(), og[n].numpy()) <= 1e-10, n
    # padding rows and the denominator: a padded step with denominator 2 * rows is half the step on its live rows alone
    pb = Problem(6, 4, True, 300, seed=9)
    idx = pb.step_indices(160, 1, True, 3)
    _, cfg = make_hyper(160, 320, True, pb.B, 0.5)
    lp, gp = pb.reference_grad(pb.p64, idx, 320, True, cfg)
    ll, gl = pb.reference_grad(pb.p64, idx[idx >= 0], 160, True, cfg)
    np.testing.assert_allclose(lp, ll * 0.5, rtol=1e-12, atol=1e-14)
    for n in pb.names:
        assert nerr(gp[n].numpy(), 0.5 * gl[n].numpy()) <= 1e-12, n


# ---------------------------------------------------------------- one step against float64 -------------------------------------
def check_one_step(pb, got, ref, max_norm, tag):
    """Returns the worst errors (gradient, loss, norm, moments, update) after asserting the bars."""
    names = pb.names
    pad = pb.padding_mask()
    errs = {}
    # losses: rtol 1e-5, atol 1e-6
    gl = got["losses"].cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(gl, ref["losses"], rtol=1e-5, atol=1e-6, err_msg=tag)
    errs["loss"] = float((np.abs(gl - ref["losses"]) / np.maximum(np.abs(ref["losses"]), 1e-6)).max())
    # pre-clip norm
    gn = float(got["gn"].cpu()[0])
    errs["norm"] = abs(gn - ref["norm"]) / ref["norm"]
    assert errs["norm"] <= 1e-5, (tag, gn, ref["norm"])
    coef = min(1.0, max_norm / (ref["norm"] + 1e-6))
    assert (coef < 1.0) == (max_norm < 1.0), (tag, "the clip case must clip and the 1e6 case must not", ref["norm"])
    # the clipped gradient of the step, per tensor, and zero padding between tensors
    G = got["G"].cpu()
    gv = pb.named64(G)
    errs["grad"] = max(nerr(gv[n].numpy(), ref["grads"][n].numpy()) for n in names)
    for n in names:
        e = nerr(gv[n].numpy(), ref["grads"][n].numpy())
        assert e <= 2e-5, (tag, n, e)
    assert float(G[pad].abs().sum()) == 0.0, tag
    # Adam moments at 1e-5 of each tensor's largest entry; parameter update within 1e-3 * lr
    mv, vv, pv, p0 = pb.named64(got["M"]), pb.named64(got["V"]), pb.named64(got["P"]), pb.named64(pb.P0)
    errs["moments"] = max(max(nerr(mv[n].numpy(), ref["M"][n].numpy()), nerr(vv[n].numpy(), ref["V"][n].numpy())) for n in names)
    assert errs["moments"] <= 1e-5, (tag, errs["moments"])
    errs["update"] = max(float(((pv[n] - p0[n]) - (ref["P"][n] - p0[n])).abs().max()) for n in names) / LR
    assert errs["update"] <= 1e-3, (tag, errs["update"])
    for t in (got["P"], got["M"], got["V"]):
        assert float(t.cpu()[pad].abs().sum()) == 0.0, tag
    return errs


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_small_update_one_step_vs_fp64(ctx, case):
    """One step on a non-zero Adam state: the clipped gradient per tensor (2e-5 of its largest entry, padding exactly 0), the four
    losses (rtol 1e-5, atol 1e-6), the pre-clip norm (rtol 1e-5), the moments (1e-5) and the parameter update (1e-3 lr) against
    float64 -- with grad_norm_clip 0.5 (clipping active) and 1e6 (coefficient 1, grads is the raw gradient)."""
    cid, D, A, cont, rows, opts, _ = case
    pb, idx, den, norm = case_setup(D, A, cont, rows, opts, 1, seed=rows * 3 + D)
    for max_norm in (0.5, 1e6):
        got = pb.run(ctx, idx, rows, 1, den, norm, max_norm)
        ref = pb.reference_update(pb.p64, pb.named64(pb.M0), pb.named64(pb.V0), idx, rows, 1, den, norm, max_norm)
        errs = check_one_step(pb, got, ref, max_norm, (cid, max_norm))
        c = plan_class(rows)
        print(f"small-net fp64 {cid} CL{c['CL']} RT{c['RT']} tiles{c['tiles']} clip {max_norm:g}: "
              + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))


# ---------------------------------------------------------------- many steps in one launch ---------------------------------------
@gpu
@pytest.mark.parametrize("case", MULTI_CASES, ids=MULTI_IDS)
def test_small_update_one_launch_equals_chained_launches(ctx, case):
    """One launch of S steps is bit-identical to S launches of one step each, every launch given its step's idx slice and
    step_consts row and chaining P / M / V: per-step losses, final P / M / V, the last step's grads and pre-clip norm.  Per step
    the arithmetic is the same; only the two-steps-ahead index / scalar prefetch and the shared-memory carry-over differ."""
    cid, D, A, cont, rows, steps, opts = case
    pb, idx, den, norm = case_setup(D, A, cont, rows, opts, steps, seed=rows + steps)
    one = pb.run(ctx, idx, rows, steps, den, norm, 0.5)
    P, M, V = pb.P0.cuda(), pb.M0.cuda(), pb.V0.cuda()
    losses = []
    for k in range(steps):
        ch = pb.run(ctx, idx[k * rows:(k + 1) * rows], rows, 1, den, norm, 0.5, P=P, M=M, V=V, t0=ADAM_T0 + k)
        losses.append(ch["losses"])
    assert torch.equal(one["losses"], torch.cat(losses)), cid
    for k in ("P", "M", "V", "G", "gn"):
        assert torch.equal(one[k], ch[k]), (cid, k)


@gpu
@pytest.mark.parametrize("case", MULTI_CASES, ids=MULTI_IDS)
def test_small_update_many_steps_vs_fp64(ctx, case):
    """The S-step launch against S sequential float64 steps (gradient -> clip -> Adam): per-step losses (rtol 1e-4), the final
    moments (1e-4 of each tensor's largest entry) and the parameter update P_S - P_0 (1e-3 lr per step, the one-step bar).  The
    update is not held to 1e-4 of its size: each step stores P in fp32, which rounds it by up to half an ulp of |P|, 6e-8 or
    2e-4 lr at |P| = 1."""
    cid, D, A, cont, rows, steps, opts = case
    pb, idx, den, norm = case_setup(D, A, cont, rows, opts, steps, seed=rows + steps)
    got = pb.run(ctx, idx, rows, steps, den, norm, 0.5)
    ref = pb.reference_update(pb.p64, pb.named64(pb.M0), pb.named64(pb.V0), idx, rows, steps, den, norm, 0.5)
    gl = got["losses"].cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(gl, ref["losses"], rtol=1e-4, atol=1e-6, err_msg=cid)
    mv, vv, pv, p0 = pb.named64(got["M"]), pb.named64(got["V"]), pb.named64(got["P"]), pb.named64(pb.P0)
    errs = dict(loss=float((np.abs(gl - ref["losses"]) / np.maximum(np.abs(ref["losses"]), 1e-6)).max()), moments=0.0, update=0.0)
    for n in pb.names:
        em = max(nerr(mv[n].numpy(), ref["M"][n].numpy()), nerr(vv[n].numpy(), ref["V"][n].numpy()))
        eu = float(((pv[n] - p0[n]) - (ref["P"][n] - p0[n])).abs().max()) / LR
        assert em <= 1e-4 and eu <= 1e-3 * steps, (cid, n, em, eu)
        errs["moments"], errs["update"] = max(errs["moments"], em), max(errs["update"], eu)
    print(f"small-net fp64 {cid} {steps} steps: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))


# ---------------------------------------------------------------- refusals ---------------------------------------------------------
@gpu
def test_small_update_refusals_then_correct(ctx):
    """rows 2049 and 0, steps 0, and networks outside the shape rule (hidden 65, act_dim 9, obs_dim 65, obs_dim 64 over the
    shared-memory budget) raise NativeError without launching or writing anything; the next valid call on the context is correct."""
    from diamond import _native as N
    from diamond.flat import FlatMlp
    pb = Problem(4, 3, False, 4200, seed=1)
    d = pb.device()
    P, M, V = pb.P0.cuda(), pb.M0.cuda(), pb.V0.cuda()
    G = torch.full((pb.fm.total,), 7.0, device="cuda")
    losses = torch.full((2, 4), 7.0, device="cuda")
    idx = dev(np.arange(4200) % pb.B, torch.int32)
    consts = dev(step_consts(ADAM_T0, 2))

    def call(desc, rows, steps, P=P, G=G, M=M, V=V):
        hyper, _ = make_hyper(max(rows, 1), max(rows, 1), False, pb.B, 0.5)
        ctx.small_update(desc, P, G, M, V, d["obs"], d["act"], d["old_lp"], d["adv"], d["ret"], None, idx, rows, steps, hyper, consts,
                         losses)

    before = [t.clone() for t in (P, M, V, G, losses)]
    n0 = ctx.launches
    for rows, steps, what in ((2049, 1, "bad shape"), (0, 1, "bad shape"), (16, 0, "bad shape")):
        with pytest.raises(N.NativeError, match=what):
            call(pb.fm.desc, rows, steps)
    for D, H, A in ((4, 65, 3), (4, 64, 9), (65, 64, 3), (64, 64, 1)):
        fm = FlatMlp(D, H, A, False)
        assert not ctx.small_update_supported(fm.desc) and not small_supported(D, H, A, False)
        z = torch.zeros(fm.total, device="cuda")
        with pytest.raises(N.NativeError, match="unsupported network"):
            call(fm.desc, 16, 1, P=z, G=z.clone(), M=z.clone(), V=z.clone())
    torch.cuda.synchronize()
    assert ctx.launches == n0
    for a, b in zip(before, (P, M, V, G, losses)):
        assert torch.equal(a, b)
    # the context keeps working: a 2-tile step against float64
    rows = 600
    idx = pb.step_indices(rows, 1, True, 5)
    got = pb.run(ctx, idx, rows, 1, rows, True, 0.5)
    ref = pb.reference_update(pb.p64, pb.named64(pb.M0), pb.named64(pb.V0), idx, rows, 1, rows, True, 0.5)
    check_one_step(pb, got, ref, 0.5, "after refusals")


# ---------------------------------------------------------------- agent level ------------------------------------------------------
def ran_small_kernel(agent):
    return any("small" in b for b in agent.engine._bufs.values())


@gpu
def test_agent_small_rows_boundary():
    """PPO takes the cluster kernel at 1024 rows per minibatch (SMALL_ROWS) and the per-layer kernels at 1025."""
    from diamond import PPO, PPOConfig, envs
    from diamond.agents import FusedMlpEngine
    assert FusedMlpEngine.SMALL_ROWS == 1024
    for N_, T, MB, small in ((32, 32, 1, True), (25, 41, 1, False)):
        rng = np.random.default_rng(N_)
        exp = [[rng.standard_normal((N_, 4)).astype(np.float32), rng.standard_normal((N_, 4)).astype(np.float32), rng.integers(0, 2, N_),
                rng.standard_normal(N_), rng.random(N_) < 0.05, rng.random(N_) < 0.05] for _ in range(T)]
        agent = PPO(lambda: envs.SyntheticEnv(4, 2), PPOConfig(num_envs=N_, rollout_steps=T, num_epochs=2, num_minibatches=MB,
                                                                verbose=False, seed=11))
        assert agent.engine.use_small_kernel
        agent.learn(exp)
        torch.cuda.synchronize()
        assert ran_small_kernel(agent) == small, N_ * T // MB
        assert agent.engine.adam_step == 2 and bool(torch.isfinite(agent.engine.P).all())
