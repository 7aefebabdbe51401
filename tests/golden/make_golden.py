"""TEST INFRASTRUCTURE ONLY — generate golden vectors by executing the UNMODIFIED reference.

Run in the build container (the only place /root/reference exists):

    python tests/golden/make_golden.py

Writes tests/golden/*.npz.  The reference has no tests or fixtures of its own
(SURVEY.md §4), so these files ARE the parity pin: every array below is an
input to, or an output of, the reference's own code (diamond/ppo.py,
diamond/continuous_ppo.py, diamond/recurrent_ppo.py) run on torch 2.11.0 /
numpy 2.3.5 CPU.  Loss components are captured with call hooks; no reference
source is edited (the recurrent case applies the documented 2-line None-check
fix, SURVEY.md §0.4).
"""
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle.ref_import import import_reference, patch_recurrent_none_checks  # noqa: E402


def synth_experience(rng, T, N, D, act, continuous, p_term=0.03, p_trunc=0.03):
    """Experience list exactly as PPO.rollout() builds it (ppo.py:165-172): per step
    [obs f32 [N,D], next_obs f32 [N,D], actions i64 [N] (f32 [N,act] continuous),
     rewards f64 [N], terminations bool [N], truncations bool [N]]."""
    exp = []
    for _ in range(T):
        obs = rng.standard_normal((N, D)).astype(np.float32)
        nobs = rng.standard_normal((N, D)).astype(np.float32)
        if continuous:
            a = rng.standard_normal((N, act)).astype(np.float32)
        else:
            a = rng.integers(0, act, size=N).astype(np.int64)
        r = rng.standard_normal(N).astype(np.float64)
        term = rng.random(N) < p_term
        trunc = (rng.random(N) < p_trunc) & ~term
        exp.append([obs, nobs, a, r, term, trunc])
    return exp


class LossHooks:
    """Records per-minibatch (policy, value, entropy, total) without editing the reference."""

    def __init__(self, continuous):
        self.rows = []
        self.cur = {}
        self.continuous = continuous

    def __enter__(self):
        self._max, self._mse, self._bwd = torch.max, torch.nn.functional.mse_loss, torch.Tensor.backward
        hooks = self
        Cat, Nrm = torch.distributions.Categorical, torch.distributions.Normal
        self._cent, self._nent = Cat.entropy, Nrm.entropy

        def max_(*a, **k):
            out = hooks._max(*a, **k)
            if len(a) == 2 and torch.is_tensor(a[1]) and out.requires_grad:   # ppo.py:270
                hooks.cur["policy"] = float(out.detach().mean())
            return out

        def mse(*a, **k):
            out = hooks._mse(*a, **k)
            if out.requires_grad:
                hooks.cur["value"] = 0.5 * float(out.detach())                          # ppo.py:272
            return out

        def cent(d):
            out = hooks._cent(d)
            if out.requires_grad:
                hooks.cur["entropy"] = float(out.detach().mean())                       # ppo.py:274
            return out

        def nent(d):
            out = hooks._nent(d)
            if out.requires_grad:
                hooks.cur["entropy"] = float(out.detach().sum(-1).mean())               # continuous_ppo.py:45-47
            return out

        def bwd(t, *a, **k):
            hooks.cur["total"] = float(t.detach())
            hooks.rows.append([hooks.cur[x] for x in ("policy", "value", "entropy", "total")])
            hooks.cur = {}
            return hooks._bwd(t, *a, **k)

        torch.max, torch.nn.functional.mse_loss, torch.Tensor.backward = max_, mse, bwd
        Cat.entropy, Nrm.entropy = cent, nent
        return self

    def __exit__(self, *exc):
        torch.max, torch.nn.functional.mse_loss, torch.Tensor.backward = self._max, self._mse, self._bwd
        torch.distributions.Categorical.entropy = self._cent
        torch.distributions.Normal.entropy = self._nent


MAX_FILE_BYTES = 1_000_000


def save_learn_fixture(name, out):
    """learn_<name>.npz; where that file would exceed 1 MB, the outputs after the last epoch go to learn_<name>.e<E>.npz
    (tests/test_agents_gpu.py load_fixture merges the two)."""
    tag = f"e{int(out['meta'][5])}."
    whole = io.BytesIO()
    np.savez_compressed(whole, **out)
    if whole.tell() > MAX_FILE_BYTES and tag != "e1.":
        np.savez_compressed(os.path.join(HERE, f"learn_{name}.{tag}npz"), **{k: v for k, v in out.items() if k.startswith(tag)})
        out = {k: v for k, v in out.items() if not k.startswith(tag)}
    np.savez_compressed(os.path.join(HERE, f"learn_{name}.npz"), **out)


def sd_np(sd, prefix):
    return {f"{prefix}{k}": v.detach().cpu().numpy().copy() for k, v in sd.items()}


def learn_case(name, kind, D, act, H, N, T, E, MB, seed_exp, save_adam=False, extra_cfg=None):
    continuous = kind == "continuous"
    diamond = import_reference(D, act, continuous)
    if continuous:
        Agent, Cfg = diamond.ContinuousPPO, diamond.ContinuousPPOConfig
    else:
        Agent, Cfg = diamond.PPO, diamond.PPOConfig
    out = {"meta": np.array([D, act, H, N, T, E, MB, int(continuous)], dtype=np.int64)}
    rng = np.random.default_rng(seed_exp)
    exp = synth_experience(rng, T, N, D, act, continuous)
    for i, key in enumerate(("obs", "next_obs", "actions", "rewards", "terminations", "truncations")):
        out[key] = np.asarray([e[i] for e in exp])

    for epochs, tag in ((1, "e1"), (E, f"e{E}")):
        kw = dict(num_envs=N, rollout_steps=T, network_hidden_dim=H, num_epochs=epochs,
                  num_minibatches=MB, verbose=False, seed=42)
        kw.update(extra_cfg or {})
        agent = Agent(lambda: None, Cfg(**kw))
        if tag == "e1":
            out.update(sd_np(agent.network.state_dict(), "init."))
        captured = {}
        orig_adv = agent.calculate_advantage

        def adv_hook(r, te, tr, v, nv):
            a = orig_adv(r, te, tr, v, nv)
            captured.update(values=v.numpy().copy(), next_values=nv.numpy().copy(), advantages=a.numpy().copy())
            return a

        agent.calculate_advantage = adv_hook
        perm_calls = []
        orig_perm = np.random.permutation

        def perm_hook(n):
            p = orig_perm(n)
            perm_calls.append(p.copy())
            return p

        np.random.seed(123)                       # SURVEY §8d: permutation seed immediately before learn()
        np.random.permutation = perm_hook
        try:
            with LossHooks(continuous) as lh:
                agent.learn(exp)
        finally:
            np.random.permutation = orig_perm
        out.update(sd_np(agent.network.state_dict(), f"{tag}.params."))
        out[f"{tag}.losses"] = np.asarray(lh.rows, dtype=np.float64)
        out[f"{tag}.lr_after"] = np.float64(agent.optimizer.param_groups[0]["lr"])
        if tag == "e1":
            out["gae.values"], out["gae.next_values"] = captured["values"], captured["next_values"]
            out["gae.advantages"] = captured["advantages"]
            out["perm0_head"] = perm_calls[0][:64].astype(np.int64)
            out["perm0_checksum"] = np.int64((perm_calls[0].astype(np.int64) * np.arange(1, len(perm_calls[0]) + 1)).sum())
            if save_adam:
                st = agent.optimizer.state_dict()["state"]
                names = [n for n, _ in agent.network.named_parameters()]
                for i, n in enumerate(names):
                    out[f"e1.exp_avg.{n}"] = st[i]["exp_avg"].numpy().copy()
                    out[f"e1.exp_avg_sq.{n}"] = st[i]["exp_avg_sq"].numpy().copy()
                    out[f"e1.step.{n}"] = np.float64(float(st[i]["step"]))
    save_learn_fixture(name, out)
    print(name, "losses[0]", out["e1.losses"][0], "n_mb", len(out["e1.losses"]))


def seeded_learn_case(name, D, act, H, N, T, E, MB, seed):
    """Large discrete fixtures (configs Smid / S, SURVEY.md 8d): inputs and initial parameters are regenerated from
    `seed` (tests/golden/seeded.py), only the reference's outputs are stored: per-minibatch losses and the 12 updated
    parameter tensors after one epoch and after E epochs, plus a thin slice of the advantages."""
    from seeded import seeded_experience, seeded_params, checksum, state_dict_of
    diamond = import_reference(D, act, False)
    obs, nobs, actions, rew, term, trunc = seeded_experience(seed, T, N, D, act)
    init = seeded_params(seed + 1, D, H, act)
    exp = [[obs[t], nobs[t], actions[t], rew[t], term[t], trunc[t]] for t in range(T)]
    out = {"meta": np.array([D, act, H, N, T, E, MB, 0], dtype=np.int64), "seed": np.int64(seed),
           "checksum": np.float64(checksum([obs, nobs, actions, rew, term, trunc] + [init[k] for k in sorted(init)]))}
    for epochs, tag in ((1, "e1"), (E, f"e{E}")):
        agent = diamond.PPO(lambda: None, diamond.PPOConfig(num_envs=N, rollout_steps=T, network_hidden_dim=H, num_epochs=epochs,
                                                            num_minibatches=MB, verbose=False, seed=42))
        agent.network.load_state_dict({k: torch.as_tensor(v) for k, v in state_dict_of(init).items()})
        captured = {}
        orig_adv = agent.calculate_advantage

        def adv_hook(r, te, tr, v, nv):
            a = orig_adv(r, te, tr, v, nv)
            captured.update(values=v.numpy()[:, :16].copy(), next_values=nv.numpy()[:, :16].copy(), advantages=a.numpy()[:, :16].copy())
            return a

        agent.calculate_advantage = adv_hook
        np.random.seed(123)
        with LossHooks(False) as lh:
            agent.learn(exp)
        out.update({k: v for k, v in sd_np(agent.network.state_dict(), f"{tag}.params.").items() if "actor_out_layer" not in k})
        out[f"{tag}.losses"] = np.asarray(lh.rows, dtype=np.float64)
        if tag == "e1":
            out["gae.values16"], out["gae.next_values16"], out["gae.advantages16"] = (captured[k] for k in ("values", "next_values", "advantages"))
    save_learn_fixture(name, out)
    print(name, "losses[0]", out["e1.losses"][0], "n_mb", len(out["e1.losses"]))


def seeded_cases():
    # the tensor-core path's shapes: minibatches of 4096 rows (Smid) and the named scale configuration itself (S: 65536-row minibatches)
    seeded_learn_case("Smid", D=64, act=4, H=256, N=256, T=128, E=4, MB=8, seed=101)
    seeded_learn_case("S", D=64, act=4, H=256, N=4096, T=128, E=4, MB=8, seed=202)


def gae_cases():
    diamond = import_reference(4, 2, False)
    out = {}
    # KAT 1 (SURVEY §8c): T=8, rewards = 1, everything else 0
    cases = {}
    T, N = 8, 2
    z = np.zeros((T, N), np.float32)
    cases["kat1"] = (np.ones((T, N), np.float32), z, z, z, z)
    # KAT 2: T=4, N=3, r=1, v=.5, nv=2; env1 terminated at t=1, env2 truncated at t=1
    T, N = 4, 3
    term = np.zeros((T, N), np.float32); term[1, 1] = 1
    trunc = np.zeros((T, N), np.float32); trunc[1, 2] = 1
    cases["kat2"] = (np.ones((T, N), np.float32), term, trunc, np.full((T, N), .5, np.float32), np.full((T, N), 2., np.float32))
    rng = np.random.default_rng(7)
    for nm, (T, N) in {"rand_small": (16, 8), "rand_ragged": (37, 45), "rand_mid": (128, 96), "t1": (1, 5)}.items():
        r = rng.standard_normal((T, N)).astype(np.float32)
        term = (rng.random((T, N)) < 0.05).astype(np.float32)
        trunc = ((rng.random((T, N)) < 0.05) & (term == 0)).astype(np.float32)
        v = rng.standard_normal((T, N)).astype(np.float32)
        nv = rng.standard_normal((T, N)).astype(np.float32)
        cases[nm] = (r, term, trunc, v, nv)
    # both masks set on the same step, and all-done rows
    T, N = 6, 4
    r = rng.standard_normal((T, N)).astype(np.float32)
    v = rng.standard_normal((T, N)).astype(np.float32); nv = rng.standard_normal((T, N)).astype(np.float32)
    term = np.zeros((T, N), np.float32); trunc = np.zeros((T, N), np.float32)
    term[2, 0] = trunc[2, 0] = 1; term[:, 1] = 1; trunc[:, 2] = 1
    cases["both_masks"] = (r, term, trunc, v, nv)
    for nm, (r, term, trunc, v, nv) in cases.items():
        T, N = r.shape
        for gam, lam, tag in ((0.99, 0.95, ""), (0.9, 0.8, ".g9l8")):
            agent = diamond.PPO(lambda: None, diamond.PPOConfig(num_envs=N, rollout_steps=T, gamma=gam, gae_lambda=lam, verbose=False))
            a = agent.calculate_advantage(*(torch.as_tensor(x) for x in (r, term, trunc, v, nv)))
            out[f"{nm}{tag}.advantages"] = a.numpy().copy()
        for k, x in zip(("rewards", "terminations", "truncations", "values", "next_values"), (r, term, trunc, v, nv)):
            out[f"{nm}.{k}"] = x
        # advantage normalisation as ppo.py:241-243
        at = torch.as_tensor(out[f"{nm}.advantages"])
        out[f"{nm}.returns"] = (torch.as_tensor(v) + at).numpy()
        if at.numel() > 1:
            out[f"{nm}.adv_norm"] = ((at - at.mean()) / (at.std() + 1e-6)).numpy()
    np.savez_compressed(os.path.join(HERE, "gae.npz"), **out)
    print("gae kat1", out["kat1.advantages"][:, 0])
    print("gae kat2", out["kat2.advantages"])


def perm_cases():
    out = {}
    for seed, n in ((42, 1024), (42, 524288), (123, 1024), (0, 1), (0, 2), (7, 1000), (5, 65537)):
        np.random.seed(seed)
        p = np.random.permutation(n)
        assert p.dtype == np.int64
        out[f"s{seed}_n{n}.head"] = p[:32].copy()
        out[f"s{seed}_n{n}.tail"] = p[-32:].copy()
        out[f"s{seed}_n{n}.checksum"] = np.int64((p * np.arange(1, n + 1)).sum())
        # the stream position after the call (next legacy draw) pins how many 32-bit words were consumed
        out[f"s{seed}_n{n}.next_u32"] = np.int64(np.random.randint(0, 2**32, dtype=np.uint64))
        if n <= 1024:
            out[f"s{seed}_n{n}.full"] = p.copy()
    # two consecutive permutations from one seed (epoch loop, ppo.py:254)
    np.random.seed(123)
    a = np.random.permutation(4096); b = np.random.permutation(4096)
    out["s123_n4096_x2.first"], out["s123_n4096_x2.second"] = a, b
    np.savez_compressed(os.path.join(HERE, "perm.npz"), **out)
    print("perm s42 n1024 head", out["s42_n1024.head"][:8])
    print("perm s42 n524288 head", out["s42_n524288.head"][:6])


def recurrent_case(name="R", D=4, A=2, H=64, Hg=16, N=8, T=16, E=2, MB=1):
    diamond = import_reference(D, A, False)
    patch_recurrent_none_checks(diamond)
    cfg = diamond.RecurrentPPOConfig(num_envs=N, rollout_steps=T, num_epochs=E, num_minibatches=MB, verbose=False,
                                     network_hidden_dim=H, gru_hidden_dim=Hg)
    agent = diamond.RecurrentPPO(lambda: None, cfg)
    out = {"meta": np.array([D, A, H, Hg, N, T, E, MB], dtype=np.int64)}
    out.update(sd_np(agent.network.state_dict(), "init."))
    rng = np.random.default_rng(11)
    # Build experience as RecurrentPPO.rollout() does (recurrent_ppo.py:214-245) with synthetic env outputs.
    torch.manual_seed(5)
    hx = torch.zeros(1, N, Hg)
    prev_dones = np.zeros(N, dtype=bool)
    exp = []
    obs = rng.standard_normal((N, D)).astype(np.float32)
    for t in range(T):
        obs_t = torch.as_tensor(obs[None], dtype=torch.float32)
        pd_t = torch.as_tensor(prev_dones[None], dtype=torch.bool)
        with torch.inference_mode():
            logits, values, new_hx = agent.network.get_logits_values_and_hx(obs_t, hx, pd_t)
        dist = torch.distributions.Categorical(logits=logits.squeeze(0))
        actions = dist.sample()
        logp = dist.log_prob(actions)
        nobs = rng.standard_normal((N, D)).astype(np.float32)
        r = rng.standard_normal(N).astype(np.float64)
        term = rng.random(N) < 0.08
        trunc = (rng.random(N) < 0.08) & ~term
        with torch.inference_mode():
            nv = agent.network.get_values(torch.as_tensor(nobs[None]), new_hx, dones=None)
        exp.append([obs_t.squeeze(0), actions, r, term, trunc, pd_t.squeeze(0), logp, values.squeeze(0), nv.squeeze(0), hx])
        dones = np.logical_or(term, trunc)
        obs = np.where(dones[:, None], rng.standard_normal((N, D)).astype(np.float32), nobs)
        hx = new_hx
        prev_dones = dones
    out["obs"] = torch.stack([e[0] for e in exp]).numpy()
    out["actions"] = torch.stack([e[1] for e in exp]).numpy()
    out["rewards"] = np.asarray([e[2] for e in exp])
    out["terminations"] = np.asarray([e[3] for e in exp])
    out["truncations"] = np.asarray([e[4] for e in exp])
    out["prev_dones"] = torch.stack([e[5] for e in exp]).numpy()
    out["log_probs"] = torch.stack([e[6] for e in exp]).numpy()
    out["values"] = torch.stack([e[7] for e in exp]).numpy()
    out["next_values"] = torch.stack([e[8] for e in exp]).numpy()
    out["hx0"] = exp[0][9].numpy().copy()
    np.random.seed(123)
    with LossHooks(False) as lh:
        agent.learn(exp)
    out.update(sd_np(agent.network.state_dict(), f"e{E}.params."))
    out[f"e{E}.losses"] = np.asarray(lh.rows, dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, f"learn_{name}.npz"), **out)
    print(name, "losses", out[f"e{E}.losses"])


def recurrent_extra_cases():
    # minibatch gather/scatter around the full-sequence BPTT (MB > 1), a GRU width off the warp-shuffle fast path, wider nets
    recurrent_case("R4", D=4, A=2, H=64, Hg=16, N=8, T=16, E=2, MB=4)
    recurrent_case("Rg", D=6, A=3, H=32, Hg=24, N=12, T=10, E=2, MB=2)
    recurrent_case("Rw", D=8, A=4, H=128, Hg=32, N=16, T=32, E=1, MB=2)


if __name__ == "__main__":
    torch.set_num_threads(1)      # deterministic summation order for the pin
    if len(sys.argv) > 1 and sys.argv[1] == "seeded":            # round 2: config S / Smid through the reference (minutes of CPU time)
        sys.path.insert(0, HERE)
        seeded_cases()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "recurrent_extra":   # added later: leaves the other fixtures untouched
        recurrent_extra_cases()
        sys.exit(0)
    gae_cases()
    perm_cases()
    learn_case("C", "discrete", D=4, act=2, H=64, N=8, T=128, E=4, MB=8, seed_exp=1, save_adam=True)
    learn_case("L", "discrete", D=8, act=4, H=64, N=8, T=128, E=4, MB=8, seed_exp=2)
    learn_case("Ssmall", "discrete", D=64, act=4, H=128, N=32, T=32, E=4, MB=8, seed_exp=3)
    learn_case("Pn", "continuous", D=3, act=1, H=64, N=64, T=64, E=4, MB=8, seed_exp=4, save_adam=True)
    learn_case("Pn3", "continuous", D=5, act=3, H=64, N=16, T=32, E=4, MB=4, seed_exp=5)
    learn_case("Cdecay", "discrete", D=4, act=2, H=64, N=8, T=32, E=2, MB=4, seed_exp=6,
               extra_cfg=dict(decay_lr=True, total_steps=8 * 32 * 10, advantage_norm=False, ppo_clip=0.1,
                              value_loss_weight=0.5, entropy_beta=0.02, grad_norm_clip=0.3, gamma=0.97, gae_lambda=0.9))
    recurrent_case()
    recurrent_extra_cases()
