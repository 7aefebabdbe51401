"""Results of the fp16-pair forward GEMMs at config S (bench.py's workload): a seeded sequence of learn() calls run three ways --
forward layers 2 and 3 on fp16 pairs (the default), the same launches forced onto 3xTF32 (tc_debug bit 2048), and the FFMA path
(tensor_cores 0).  Prints, per loss column and parameter tensor, the largest relative difference of fp16 pairs against TF32 and of
TF32 against FFMA, and exits non-zero if the first exceeds the second anywhere (beyond fp32 rounding of the largest element).

Needs a B200 and a library built with timing switches:  make -C diamond-ppo_b200 EXTRA=-DDPPO_TIMING_SWITCHES
  python tests/fp16_pair_parity.py [--pkg DIR] [--learns N] [--out FILE]
--pkg: the directory that holds the `diamond` package of that build (default: this tree's)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pkg", default=os.path.join(ROOT, "diamond-ppo_b200"))
    ap.add_argument("--learns", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.abspath(args.pkg))
    import numpy as np
    import torch
    from diamond import PPO, PPOConfig, envs, _native          # before bench, which puts this tree's package on sys.path
    from diamond.agents import RolloutBuffer
    import bench

    ctx = _native.get_context(0)

    def env_fn(n):
        return envs.BatchedSyntheticVectorEnv(n, bench.D, bench.A)
    env_fn.vectorized = True
    host = bench.synth_host_rollout(1)

    def run(tensor_cores, tc_debug):
        ctx.set_option("tensor_cores", tensor_cores)
        ctx.set_option("tc_debug", tc_debug)
        cfg = PPOConfig(num_envs=bench.N_ENVS, rollout_steps=bench.T, network_hidden_dim=bench.H, num_epochs=bench.E,
                        num_minibatches=bench.MB, verbose=False, total_steps=bench.T * bench.N_ENVS * 1000, seed=7)
        agent = PPO(env_fn, cfg)
        buf = RolloutBuffer(ctx, bench.T, bench.N_ENVS, bench.D, 1, False, agent.device)
        buf.load_host(*host)
        np.random.seed(123)
        losses = []
        for _ in range(args.learns):
            agent.learn(buf)
            losses.append(agent.last_losses.cpu().numpy())
        torch.cuda.synchronize()
        out = {f"losses[:, {i}]": np.stack(losses)[..., i] for i in range(4)}
        out.update({n: p.detach().cpu().numpy() for n, p in agent.network.named_parameters()})
        ctx.set_option("tensor_cores", 1)
        ctx.set_option("tc_debug", 0)
        return out

    f16, tf32, ffma = run(1, 0), run(1, 2048), run(0, 0)

    def rel(a, b):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))

    rows, ok = {}, True
    for k in f16:
        r = {"f16_vs_tf32": rel(f16[k], tf32[k]), "tf32_vs_ffma": rel(tf32[k], ffma[k])}
        r["ok"] = r["f16_vs_tf32"] <= max(r["tf32_vs_ffma"], 2.0 ** -23)
        ok &= r["ok"]
        rows[k] = r
        print(f"{k:32s} fp16 pairs vs TF32 {r['f16_vs_tf32']:.3e}   TF32 vs FFMA {r['tf32_vs_ffma']:.3e}   {'ok' if r['ok'] else 'LARGER'}")
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"learns": args.learns, "ok": ok, "arrays": rows}, f, indent=1)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
