"""CPU: pins the oracle (oracle/ppo_oracle.py, oracle/oracle.c) against golden vectors produced by the
unmodified reference (tests/golden/make_golden.py).  The reference itself ships no tests (SURVEY.md §4)."""
import os

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as O
from oracle import c_oracle as C

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
GAE_CASES = ["kat1", "kat2", "rand_small", "rand_ragged", "rand_mid", "t1", "both_masks"]


def _load(name):
    return np.load(os.path.join(GOLDEN, name))


def test_gae_kats_hand_checkable():
    g = _load("gae.npz")
    # SURVEY §8c KAT 1: sum_k (gamma*lambda)^k
    gl = 0.99 * 0.95
    expect = [sum(gl ** k for k in range(n)) for n in range(8, 0, -1)]
    np.testing.assert_allclose(g["kat1.advantages"][:, 0], expect, rtol=1e-6)
    np.testing.assert_allclose(g["kat2.advantages"],
                               [[9.069237, 2.950250, 4.812440], [7.006100, 0.5, 2.48], [4.812440] * 3, [2.48] * 3], rtol=1e-6)


@pytest.mark.parametrize("case", GAE_CASES)
@pytest.mark.parametrize("tag,gam,lam", [("", 0.99, 0.95), (".g9l8", 0.9, 0.8)])
def test_gae_oracles_bit_exact(case, tag, gam, lam):
    g = _load("gae.npz")
    args = [g[f"{case}.{k}"] for k in ("rewards", "terminations", "truncations", "values", "next_values")]
    ref = g[f"{case}{tag}.advantages"]
    np.testing.assert_array_equal(O.gae(*args, gam, lam), ref)           # numpy restatement: bit-exact
    adv, ret = C.gae(*args, gam, lam)
    np.testing.assert_array_equal(adv, ref)                                # C restatement: bit-exact
    if tag == "":
        np.testing.assert_array_equal(ret, g[f"{case}.returns"])


@pytest.mark.parametrize("case", [c for c in GAE_CASES if c != "t1"])
def test_adv_norm(case):
    g = _load("gae.npz")
    ret, an = O.returns_and_normalise(g[f"{case}.values"], g[f"{case}.advantages"], True)
    np.testing.assert_array_equal(ret, g[f"{case}.returns"])
    ref = g[f"{case}.adv_norm"]
    assert np.abs(an - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())


def test_permutation_oracles_bit_exact():
    g = _load("perm.npz")
    for seed, n in ((42, 1024), (123, 1024), (0, 1), (0, 2), (7, 1000)):
        p = O.legacy_permutation(O.MT19937(seed), n)
        np.testing.assert_array_equal(p, g[f"s{seed}_n{n}.full"])
    for seed, n in ((42, 1024), (42, 524288), (123, 1024), (0, 1), (0, 2), (7, 1000), (5, 65537)):
        mt = C.MT(seed)
        p = mt.permutation(n)
        np.testing.assert_array_equal(p[:32], g[f"s{seed}_n{n}.head"])
        np.testing.assert_array_equal(p[-32:], g[f"s{seed}_n{n}.tail"])
        assert int((p * np.arange(1, n + 1)).sum()) == int(g[f"s{seed}_n{n}.checksum"])
        assert sorted(p.tolist()) == list(range(n)) if n <= 65537 else True
        assert mt.next_u32() == int(g[f"s{seed}_n{n}.next_u32"])        # stream position after the call
    mt = C.MT(123)
    np.testing.assert_array_equal(mt.permutation(4096), g["s123_n4096_x2.first"])
    np.testing.assert_array_equal(mt.permutation(4096), g["s123_n4096_x2.second"])
    # and against the live numpy in this image
    np.random.seed(99)
    np.testing.assert_array_equal(C.MT(99).permutation(5000), np.random.permutation(5000))


def _run_learn(name, epochs_tag, extra=None):
    g = _load(f"learn_{name}.npz")
    D, act, H, N, T, E, MB, cont = (int(x) for x in g["meta"])
    cont = bool(cont)
    names = O.CONTINUOUS_PARAM_NAMES if cont else O.DISCRETE_PARAM_NAMES
    p = {n: torch.as_tensor(g[f"init.{n}"]).clone() for n in names}
    state = O.new_adam_state(p, names)
    epochs = int(epochs_tag[1:])
    cfg = O.default_cfg(num_epochs=epochs, num_minibatches=MB, **(extra or {}))
    mt = C.MT(123)
    perms = np.stack([mt.permutation(T * N) for _ in range(epochs)])
    losses, inter = O.learn(p, state, g["obs"], g["next_obs"], g["actions"], g["rewards"], g["terminations"],
                            g["truncations"], cfg, perms, continuous=cont)
    return g, p, state, losses, inter, names


@pytest.mark.parametrize("name", ["C", "L", "Ssmall", "Pn", "Pn3"])
def test_learn_oracle_one_epoch(name):
    g, p, state, losses, inter, names = _run_learn(name, "e1")
    # GAE is bit-exact on the reference's own values.  The oracle's values come from the host's float32 GEMMs, whose rounding
    # depends on the CPU's instruction set (MKL picks its kernels per CPU), so they and the advantages computed from them are
    # compared to a tolerance.
    rollout = [np.asarray(g[k]).astype(np.float32) for k in ("rewards", "terminations", "truncations")]
    cfg = O.default_cfg()
    np.testing.assert_array_equal(O.gae(*rollout, g["gae.values"], g["gae.next_values"], cfg["gamma"], cfg["gae_lambda"]),
                                  g["gae.advantages"])
    assert np.abs(inter["advantages"] - g["gae.advantages"]).max() / np.abs(g["gae.advantages"]).max() <= 1e-5
    np.testing.assert_allclose(inter["values"], g["gae.values"], rtol=1e-5, atol=1e-6)
    ref_l = g["e1.losses"]
    got = np.array([[l[k] for k in ("policy", "value", "entropy", "total")] for l in losses])
    np.testing.assert_allclose(got, ref_l, rtol=1e-4, atol=2e-6)
    for n in names:
        ref = g[f"e1.params.{n}"]
        err = np.abs(p[n].numpy() - ref).max() / max(np.abs(ref).max(), 1e-12)
        assert err <= 1e-5, (n, err)
    if f"e1.exp_avg.{names[0]}" in g:
        for n in names:
            np.testing.assert_allclose(state["exp_avg"][n].numpy(), g[f"e1.exp_avg.{n}"], rtol=1e-4, atol=1e-8)
            np.testing.assert_allclose(state["exp_avg_sq"][n].numpy(), g[f"e1.exp_avg_sq.{n}"], rtol=1e-4, atol=1e-12)


def test_learn_oracle_one_epoch_config_Smid_seeded():
    """The oracle at the tensor-core path's shapes (H = 256, 4096-row minibatches) against the reference's outputs on the seeded
    inputs of tests/golden/seeded.py (the same fixture the GPU parity test of config S uses)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from seeded import seeded_experience, seeded_params, checksum
    g = _load("learn_Smid.npz")
    D, act, H, N, T, E, MB, _ = (int(x) for x in g["meta"])
    seed = int(g["seed"])
    obs, nobs, actions, rew, term, trunc = seeded_experience(seed, T, N, D, act)
    init = seeded_params(seed + 1, D, H, act)
    assert checksum([obs, nobs, actions, rew, term, trunc] + [init[k] for k in sorted(init)]) == float(g["checksum"])
    names = O.DISCRETE_PARAM_NAMES
    p = {n: torch.as_tensor(init[n]).clone() for n in names}
    state = O.new_adam_state(p, names)
    mt = C.MT(123)
    perms = np.stack([mt.permutation(T * N)])
    losses, inter = O.learn(p, state, obs, nobs, actions, rew, term, trunc, O.default_cfg(num_epochs=1, num_minibatches=MB), perms)
    assert np.abs(inter["advantages"][:, :16] - g["gae.advantages16"]).max() / np.abs(g["gae.advantages16"]).max() <= 1e-5
    got = np.array([[l[k] for k in ("policy", "value", "entropy", "total")] for l in losses])
    np.testing.assert_allclose(got, g["e1.losses"], rtol=1e-4, atol=5e-6)
    for n in names:
        ref = g[f"e1.params.{n}"]
        err = np.abs(p[n].numpy() - ref).max() / max(np.abs(ref).max(), 1e-12)
        assert err <= 1e-4, (n, err)


@pytest.mark.parametrize("name", ["C", "Pn"])
def test_learn_oracle_four_epochs(name):
    g, p, state, losses, inter, names = _run_learn(name, "e4")
    got = np.array([[l[k] for k in ("policy", "value", "entropy", "total")] for l in losses])
    np.testing.assert_allclose(got, g["e4.losses"], rtol=2e-4, atol=5e-6)
    for n in names:
        ref = g[f"e4.params.{n}"]
        err = np.abs(p[n].numpy() - ref).max() / max(np.abs(ref).max(), 1e-12)
        assert err <= 1e-4, (n, err)


def test_learn_oracle_nondefault_cfg_and_lr_decay():
    extra = dict(advantage_norm=False, ppo_clip=0.1, value_loss_weight=0.5, entropy_beta=0.02, grad_norm_clip=0.3,
                 gamma=0.97, gae_lambda=0.9)
    g, p, state, losses, inter, names = _run_learn("Cdecay", "e1", extra)
    got = np.array([[l[k] for k in ("policy", "value", "entropy", "total")] for l in losses])
    np.testing.assert_allclose(got, g["e1.losses"], rtol=1e-4, atol=2e-6)
    for n in names:
        ref = g[f"e1.params.{n}"]
        assert np.abs(p[n].numpy() - ref).max() / max(np.abs(ref).max(), 1e-12) <= 1e-5
    # LinearLR after one learn(): total_iters = total_steps // (N*T) = 10, end factor 0.05 (ppo.py:137-142,287)
    assert abs(3e-4 * O.linear_lr_factor(1, 10, 1.0, 0.05) - float(g["e1.lr_after"])) < 1e-12


def test_gru_restatement_matches_nn_gru():
    torch.manual_seed(0)
    gru = torch.nn.GRU(6, 5)
    p = {f"gru.{k}": v.detach() for k, v in gru.named_parameters()}
    x = torch.randn(7, 3, 6)
    h0 = torch.randn(3, 5)
    dones = torch.zeros(7, 3, dtype=torch.bool)
    out, h = O.gru_forward(p, x, h0, dones)
    ref_out, ref_h = gru(x, h0.unsqueeze(0))
    np.testing.assert_allclose(out.numpy(), ref_out.detach().numpy(), atol=1e-6)
    np.testing.assert_allclose(h.numpy(), ref_h[0].detach().numpy(), atol=1e-6)


def test_recurrent_core_matches_stepwise_nn_gru():
    """GRUCore (one input-projection GEMM + T hidden steps, functional done-masking) equals the reference's loop of one-step
    nn.GRU calls with in-place hidden resets (recurrent_ppo.py:82-87, with the documented `is None` fix), values and gradients."""
    import torch
    from diamond.recurrent import GRUCore
    torch.manual_seed(0)
    T, B, H, Hg = 9, 5, 12, 7
    core = GRUCore(H, Hg)
    x = torch.randn(T, B, H, requires_grad=True)
    hx0 = torch.randn(1, B, Hg)
    dones = torch.rand(T, B) < 0.3
    out, hT = core.forward(x, hx0.clone(), dones)
    # reference-style evaluation
    x2 = x.detach().clone().requires_grad_(True)
    h = hx0.clone()
    outs = []
    for t in range(T):
        h = h.clone()
        h[:, dones[t]] = 0.0
        o, h = torch.nn.GRU.forward(core, x2[t:t + 1], h)
        outs.append(o)
    ref = torch.cat(outs, 0)
    assert torch.allclose(out, ref, atol=1e-6) and torch.allclose(hT, h, atol=1e-6)
    w = torch.randn_like(out)
    g1 = torch.autograd.grad((out * w).sum(), [x] + list(core.parameters()))
    g2 = torch.autograd.grad((ref * w).sum(), [x2] + list(core.parameters()))
    for a, b in zip(g1, g2):
        assert torch.allclose(a, b, atol=2e-6)
    # None handling (the reference's `or` raises here)
    o3, _ = core.forward(x.detach(), None, None)
    assert o3.shape == (T, B, Hg)


def test_env_oracle_matches_per_env_host_implementation():
    """oracle/env_oracle.py (vectorised restatement of Gymnasium's CartPole-v1 / Pendulum-v1 steps) against the independent
    per-environment host classes in diamond/envs.py, plus a hand-computed CartPole step."""
    from diamond import envs
    from oracle import env_oracle as EO
    rng = np.random.default_rng(0)
    # hand-computed: state 0, action 1 -> temp = 10/1.1, th_acc = -temp / (0.5 (4/3 - 0.1/1.1)), x_acc = temp - 0.05 th_acc / 1.1
    nxt, obs, r, term, trunc = EO.cartpole_step(np.zeros((1, 4)), np.array([1]), np.array([0]))
    temp = 10.0 / 1.1
    th_acc = -temp / (0.5 * (4.0 / 3.0 - 0.1 / 1.1))
    np.testing.assert_allclose(nxt[0], [0.0, 0.02 * (temp - 0.05 * th_acc / 1.1), 0.0, 0.02 * th_acc], rtol=1e-14)
    assert r[0] == 1.0 and not term[0] and not trunc[0]
    for _ in range(200):
        e = envs.CartPoleEnv()
        e.state = rng.uniform(-1, 1, 4) * np.array([2.6, 2.0, 0.25, 2.0])
        e.t = int(rng.integers(0, 500))
        s0, t0, a = e.state.copy(), e.t, int(rng.integers(0, 2))
        o, rew, te, tr, _ = e.step(a)
        nxt, obs, r, term, trunc = EO.cartpole_step(s0[None], np.array([a]), np.array([t0]))
        np.testing.assert_allclose(nxt[0], e.state, rtol=1e-13, atol=1e-15)
        np.testing.assert_array_equal(obs[0], o)
        assert (bool(term[0]), bool(trunc[0]), float(r[0])) == (te, tr, rew)
        p = envs.PendulumEnv()
        p.th, p.thdot, p.t = float(rng.uniform(-7, 7)), float(rng.uniform(-8, 8)), int(rng.integers(0, 200))
        s0, t0, u = np.array([[p.th, p.thdot]]), p.t, rng.uniform(-3, 3, (1, 1)).astype(np.float32)
        o, rew, te, tr, _ = p.step(u[0])
        nxt, obs, r, term, trunc = EO.pendulum_step(s0, u, np.array([t0]))
        np.testing.assert_allclose(nxt[0], [p.th, p.thdot], rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(obs[0], o, rtol=0, atol=1e-7)
        assert abs(r[0] - rew) <= 1e-12 * max(1.0, abs(rew)) and bool(trunc[0]) == tr and not te
