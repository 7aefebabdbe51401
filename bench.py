#!/usr/bin/env python
"""Benchmark of the Diamond PPO hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[4], "synthetic scale"): ONE 4096-env x 128-step buffer, obs_dim 64, default actor-critic
MLP at hidden 256, 4 actions, 4 epochs x 8 minibatches.  A "step" is one PPO.learn() over that buffer: pre-update pass,
GAE, advantage statistics, 32 optimiser steps.  With --gpus N the buffer is env-sharded over the N ranks (rank r owns envs
[r*4096/N, (r+1)*4096/N), STRONG scaling) and every rank holds the reference's global permutation, so the N-GPU update
is the single-GPU update up to fp32 summation order; the round-1 weak-scaling measurement (4096 envs per GPU) is kept
as the extra key `weak_scaling`.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "diamond-ppo_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

T, N_ENVS, D, H, A, E, MB = 128, 4096, 64, 256, 4, 4, 8
FLOP_PER_SAMPLE_UPDATE = 1_252_864          # SURVEY.md §8d: 2*(3F - D*H), F = D*H + 3H^2 + H*A + H
FLOP_PER_SAMPLE_PREPASS = 723_968           # 2*(F + Fc)
GAE_BYTES_PER_ELEM = 28                     # 5 fp32 reads + 2 fp32 writes
# dram__bytes_read.sum + dram__bytes_write.sum of one tc3_gemm_kernel launch at this shape (ncu --set full, cold caches,
# profiles/r4i_kernels.csv): 67.8 MB read + 10.4 MB written before the kernel ends (the rest of the 67 MB output is still in L2;
# round 1, with the next-tile L2 prefetch: 84.2 MB).  In situ (caches not flushed between the launches of an optimiser step) the same
# launch reads 6-11 MB from DRAM -- its input is its predecessor's output (profiles/r4d_insitu_traffic.md).
GEMM_DRAM_TRAFFIC = 78.1e6
# one gae_pipe_kernel launch on a cold buffer set (profiles/r1f_gae_kernels.csv): 10.5 MB read; the 4.2 MB of advantages / returns are
# still in L2 when the kernel ends (dram__bytes_write.sum = 0) and reach DRAM by eviction as the benchmark cycles its 20 buffer sets
GAE_DRAM_TRAFFIC = 10.5e6


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons while the timed region runs (NVML; nvidia-smi semantics)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_sm = index, threading.Event(), [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {getattr(nv, k): k for k in dir(nv) if k.startswith("nvmlClocksEventReason") or k.startswith("nvmlClocksThrottleReason")}
        while not self.stop_flag.is_set():
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if isinstance(bit, int) and bit and (mask & bit) and "None" not in name and "All" not in name:
                        self.reasons.add(name.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", ""))
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        self.stop_flag.set()
        self.join(timeout=1.0)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(r for r in self.reasons if r not in ("GpuIdle", "ApplicationsClocksSetting"))}


def synth_host_rollout(seed, envs=None, pin=True):
    """Synthetic rollout of config S in the buffer's dtypes (SURVEY.md 8d); envs = (lo, hi) keeps that env range of the 4096."""
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(T, N_ENVS, D, generator=g)
    next_obs = torch.randn(T, N_ENVS, D, generator=g)
    actions = torch.randint(0, A, (T, N_ENVS), generator=g, dtype=torch.int32)
    rewards = torch.randn(T, N_ENVS, generator=g)
    term = (torch.rand(T, N_ENVS, generator=g) < 0.01).float()
    trunc = ((torch.rand(T, N_ENVS, generator=g) < 0.01) & (term == 0)).float()
    out = [obs, next_obs, actions, rewards, term, trunc]
    if envs is not None:
        out = [x[:, envs[0]:envs[1]].contiguous() for x in out]
    pin = pin and torch.cuda.is_available()               # the reference arm also runs on hosts without a GPU
    return [x.pin_memory() if pin else x for x in out]


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of the reference's learn() on the host cores
# ---------------------------------------------------------------------------------------------
CPU_SAMPLE_ENVS = 512


def cpu_reference(steps, warmup, sample_envs=CPU_SAMPLE_ENVS):
    """Each step = ONE WHOLE learn() of the oracle port (oracle/ppo_oracle.py: tensorisation, pre-update pass, GAE, returns +
    normalisation, np.random permutations, 4 epochs x 8 minibatches of forward / loss / backward / clip / Adam; ppo.py:224-287)
    on a bounded sample of the workload: the first `sample_envs` of the 4096 envs (all 128 steps), i.e. minibatches of
    sample_envs*128/8 rows at the same network size.  Throughput is per sample-update, the same unit as the GPU arm."""
    from oracle import ppo_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    host = synth_host_rollout(1, envs=(0, sample_envs), pin=False)
    obs, nobs, act, rew, term, trunc = (x.numpy() for x in host)
    from diamond.networks import ActorCriticNetwork, network_parameter_init_
    from diamond.config import PPOConfig
    from diamond import envs
    torch.manual_seed(42)
    cfg = PPOConfig(network_hidden_dim=H)
    net = ActorCriticNetwork(envs.Box(shape=(D,)), envs.Discrete(A), cfg)
    network_parameter_init_(net, gain=2 ** 0.5)
    p = {n: q.detach().clone() for n, q in net.named_parameters()}
    names = O.DISCRETE_PARAM_NAMES
    state = O.new_adam_state(p, names)
    ocfg = O.default_cfg(num_epochs=E, num_minibatches=MB)
    B = T * sample_envs
    np.random.seed(123)
    t_gae = []

    def step():
        perms = np.stack([np.random.permutation(B) for _ in range(E)])              # ppo.py:252-255
        O.learn(p, state, obs, nobs, act.astype(np.int64), rew.astype(np.float64), term != 0, trunc != 0, ocfg, perms)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    # GAE alone (the reference's reverse time loop, ppo.py:188-222) on the full 4096 x 128 shape, for the GB/s line
    full = synth_host_rollout(1, pin=False)
    v, nv = np.random.standard_normal((2, T, N_ENVS)).astype(np.float32)
    t1 = time.perf_counter()
    O.gae(full[3].numpy(), full[4].numpy(), full[5].numpy(), v, nv)
    t_gae = time.perf_counter() - t1
    samples = steps * E * B
    return dict(value=samples / dt, ms_per_step=dt / steps * 1e3, cores=cores, t_gae_s=t_gae,
                gae_gbps=T * N_ENVS * GAE_BYTES_PER_ELEM / t_gae / 1e9,
                sample=f"each step = one whole learn() (pre-update pass, GAE, normalisation, {E} numpy permutations, {E} x {MB} optimiser "
                       f"steps) of the oracle port on the first {sample_envs} of the {N_ENVS} envs x {T} steps ({B // MB}-row minibatches, "
                       f"same network); ms_per_step is for that {sample_envs}/{N_ENVS} sample")


def run_reference(args, rank, world):
    if rank != 0:
        return
    r = cpu_reference(args.steps, args.warmup)
    line = {"impl": "reference", "metric": "ppo_update_samples_per_s", "value": r["value"], "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(1),
            "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                             "gae_gbps": r["gae_gbps"]},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(world):
    return {"workload": f"synthetic scale (BASELINE.json configs[4]): {N_ENVS} envs x {T} steps, obs_dim {D}, "
                        f"2x{H} trunk + {H}-wide heads, {A} actions, {E} epochs x {MB} minibatches",
            "envs_total": N_ENVS, "envs_per_gpu": N_ENVS // world, "rollout_steps": T, "global_batch": T * N_ENVS,
            "minibatch": T * N_ENVS // MB, "parallelism": f"env-sharded dp{world} (strong scaling of the one buffer)" if world > 1 else "single GPU",
            "permutation": ("bit-exact numpy MT19937 stream (host thread, overlapped)" if world == 1 else
                            "the reference's GLOBAL permutation on every rank (bit-exact numpy MT19937 stream, host thread); a device "
                            "kernel keeps each rank's members per minibatch, padded to fixed step shapes"),
            "exchange": None if world == 1 else "per optimiser step: one fused kernel per rank sums all ranks' gradients over NVLink peer "
                                                "memory (rank order) + global-norm partials, then clip + Adam",
            "l2": "inputs (2 x 134 MB observations at 1 GPU) exceed the 126 MB L2; GAE sub-benchmark cycles 20 buffer sets (294 MB)"}


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def bench_gae(ctx, hbm_peak, sets=20, launches=200, settled=True, n_envs=None):
    f = dict(device="cuda", dtype=torch.float32)
    N_ENVS = n_envs or globals()["N_ENVS"]
    bufs = []
    for s in range(sets):
        r, v, nv = (torch.randn(T, N_ENVS, **f) for _ in range(3))
        te = (torch.rand(T, N_ENVS, device="cuda") < 0.01).float()
        tr = ((torch.rand(T, N_ENVS, device="cuda") < 0.01) & (te == 0)).float()
        bufs.append((r, te, tr, v, nv, torch.empty(T, N_ENVS, **f), torch.empty(T, N_ENVS, **f)))
    for i in range(2 * sets):
        b = bufs[i % sets]
        ctx.gae(*b[:5], 0.99, 0.95, advantages=b[5], returns=b[6], inputs_settled=settled)
    torch.cuda.synchronize()
    # `launches` back-to-back launches cycling through the buffer sets (consecutive launches touch disjoint buffers, so the
    # "inputs settled" promise of include/dppo.h holds), replayed as one CUDA graph so that the host-side launch cost of
    # the Python binding does not enter the per-launch device time
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            for i in range(launches):
                b = bufs[i % sets]
                ctx.gae(*b[:5], 0.99, 0.95, advantages=b[5], returns=b[6], inputs_settled=settled)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / launches
    bytes_ = T * N_ENVS * GAE_BYTES_PER_ELEM
    gbps = bytes_ / (us * 1e-6) / 1e9
    return {"us_per_launch": us, "achieved": gbps, "peak": hbm_peak, "unit": "GB/s", "frac": gbps / hbm_peak, "bound": "hbm",
            "bytes_per_launch": bytes_, "launches": launches, "buffer_sets": sets, "inputs_settled": settled}


def bench_dominant_gemm(ctx, tensor_peak, sets=4, reps=12):
    """The dominant kernel of the update loop, timed alone with CUDA events: the CTA-pair tcgen05 GEMM at the trunk-layer
    shape of one minibatch ([65536, 256] x [256, 256]^T, bias + tanh epilogue).  `sets` rotating input/output pairs
    (4 x 134 MB > the 126 MB L2) keep the operands HBM-resident; the weight images are prepared once (they are
    L2-resident in the real step too)."""
    M, K, N = T * N_ENVS // MB, H, H
    g = torch.Generator(device="cuda").manual_seed(7)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    ins = [torch.randn(M, K, device="cuda", generator=g) for _ in range(sets)]
    outs = [torch.empty(M, N, device="cuda") for _ in range(sets)]
    ws = torch.empty(ctx.lib.dppo_tc_linear_workspace_bytes(N, K), device="cuda", dtype=torch.uint8)
    ctx.tc_linear(1, ins[0], W, False, bias=b, out=outs[0], ws=ws)
    for i in range(sets):
        ctx.tc_linear(1, ins[i], W, False, bias=b, out=outs[i], ws=ws, prepared=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        ctx.tc_linear(1, ins[i % sets], W, False, bias=b, out=outs[i % sets], ws=ws, prepared=True)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    flops = 2.0 * M * N * K
    tf = flops / (us * 1e-6) / 1e12
    return {"bound": "tensor", "kernel": "tc3_gemm_kernel<BIAS_TANH> (3xTF32 tcgen05 cta_group::2), layer base.2 of one minibatch: "
                                         f"[{M},{K}] x [{N},{K}]^T", "us_per_launch": us, "flops_per_launch": flops,
            "achieved": tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": tf / tensor_peak,
            "bytes_per_launch": 4.0 * M * (K + N), "launches": reps, "buffer_sets": sets}


def bench_mma_probe(ctx):
    """SM cycles per tcgen05.mma (M=256 over a CTA pair, N=256, K=8 tf32, shared-memory operands) on every SM pair."""
    c = ctx.mma_probe(1, 0, 256, 4000)
    return float(c.mean())


def bench_fma_peak(ctx):
    sink = torch.ones(128, device="cuda")
    iters = 1 << 16
    ctx.fma_peak(sink, iters)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        blocks, threads = ctx.fma_peak(sink, iters)
    e1.record()
    torch.cuda.synchronize()
    flops = 5 * 2.0 * iters * blocks * threads
    return flops / (e0.elapsed_time(e1) * 1e-3) / 1e12


def bench_train_iteration(reps=3):
    """One full training iteration of config S with the environments on the device (diamond/envs.py DeviceVectorEnv, synthetic
    shape stand-in): rollout() (sampling kernel + environment kernel per step, nothing crosses PCIe, log-probs / values recorded)
    followed by learn() (which then skips the pre-update pass).  Wall clock around synchronised iterations."""
    from diamond import PPO, PPOConfig
    from diamond.envs import DeviceVectorEnv
    cfg = PPOConfig(num_envs=N_ENVS, rollout_steps=T, network_hidden_dim=H, num_epochs=E, num_minibatches=MB, verbose=False,
                    total_steps=T * N_ENVS * 1000, seed=1)
    agent = PPO(DeviceVectorEnv.factory("Synthetic", obs_dim=D, n_actions=A, seed=1), cfg)
    agent.ticker = None
    agent.current_observations, _ = agent.envs.reset(seed=1)
    for _ in range(3):
        agent.learn(agent.rollout())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        buf = agent.rollout()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    for _ in range(reps):
        agent.learn(agent.rollout())
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    ms_roll, ms_iter = (t1 - t0) * 1e3 / reps, (t2 - t1) * 1e3 / reps
    return {"workload": "device-resident synthetic envs: rollout() + learn() per iteration, config S", "rollout_ms": ms_roll,
            "iteration_ms": ms_iter, "env_steps_per_s": T * N_ENVS / (ms_iter * 1e-3), "rollout_env_steps_per_s": T * N_ENVS / (ms_roll * 1e-3),
            "sample_updates_per_s": E * T * N_ENVS / (ms_iter * 1e-3)}


def learn_outputs(agent):
    """What learn() leaves its caller: the per-minibatch losses [E*MB, 4] (policy, value, entropy, total) and the updated
    network parameters."""
    out = {"losses": agent.last_losses.cpu().numpy()}
    out.update({f"params.{n}": p.detach().cpu().numpy() for n, p in agent.network.named_parameters()})
    return out


def time_learn(agent, buf, host, steps, warmup, world, dist, ctx, keep_outputs=False):
    """(ms per learn() device-resident, per-phase ms, launches, clocks, ms per learn() end to end, h2d bytes, losses).
    keep_outputs: also return learn_outputs() of the last timed learn(), read after the timed region."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        agent.learn(buf)
    barrier()
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    launches0 = ctx.launches
    ev_all = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ev = {}
        agent.learn(buf, events=ev)
        ev_all.append(ev)
    e1.record()
    barrier()
    launches = ctx.launches - launches0
    clocks = sampler.result()
    ms_total = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    phases = {"prepass": float(np.mean([ev["start"].elapsed_time(ev["prepass_end"]) for ev in ev_all])),
              "gae_and_stats": float(np.mean([ev["prepass_end"].elapsed_time(ev["gae_end"]) for ev in ev_all])),
              "update_loop": float(np.mean([ev["gae_end"].elapsed_time(ev["update_end"]) for ev in ev_all]))}
    out = dict(ms=float(ms_total) / steps, phases=phases, launches=launches, clocks=clocks)
    if keep_outputs:
        out["outputs"] = learn_outputs(agent)
    if host is None:
        return out
    # ---- end to end through the public API with host buffers ----
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h_losses = [torch.empty(E * MB, 4).pin_memory() for _ in range(2)]
    read_done = [None, None]
    # Two device buffers: the host -> device copy of step k+1's inputs is issued as soon as learn(k) has been enqueued and runs on
    # the copy stream under step k's update loop (every step's inputs are copied and every step's losses are read inside the
    # timed region; only the first copy is exposed).
    bufs = [buf, type(buf)(ctx, buf.T, buf.N, buf.D, buf.A, buf.continuous, buf.device)]
    for b_ in bufs:                                   # both buffers seen once: graph capture of the update loop outside the timed region
        b_.load_host(*host)
        agent.learn(b_)
        agent.learn(b_)
    barrier()
    e0.record()
    h2d = bufs[0].load_host(*host)                    # step 0's inputs: pinned host -> device
    for k in range(steps):
        cur = bufs[k & 1]
        agent.learn(cur)
        if k + 1 < steps:
            bufs[(k + 1) & 1].load_host(*host)        # next step's inputs, overlapped with this step's update loop
        h_losses[k & 1].copy_(agent.last_losses, non_blocking=True)      # this step's result read back (asynchronously) ...
        read_done[k & 1] = torch.cuda.Event()
        read_done[k & 1].record()
        if k > 0:
            read_done[(k - 1) & 1].synchronize()                          # ... and consumed one step later: the host never idles the GPU
            assert torch.isfinite(h_losses[(k - 1) & 1]).all()
    read_done[(steps - 1) & 1].synchronize()
    e1.record()
    barrier()
    ms_e2e = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_e2e, op=dist.ReduceOp.MAX)
    assert torch.isfinite(h_losses[(steps - 1) & 1]).all()
    out.update(ms_e2e=float(ms_e2e) / steps, h2d=int(h2d), d2h=int(h_losses[0].numel() * 4))
    return out


def dump_outputs(path, arrays):
    """DIR/<name>.npy per array, float32 or float64, so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, f"{name}.npy"), a)


def replicas_identical(agent, dist):
    flat = agent.engine.P.clone()
    ref = flat.clone()
    dist.broadcast(ref, src=0)
    ok = torch.tensor([int(torch.equal(flat, ref) and bool(torch.isfinite(flat).all()))], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return bool(int(ok))


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from diamond import PPO, PPOConfig, envs, _native
    from diamond.agents import RolloutBuffer
    torch.cuda.set_device(local_rank)
    ctx = _native.get_context(local_rank)
    hbm_peak, bf16_peak, peak_src = measured_peaks()
    if N_ENVS % world != 0:
        raise SystemExit(f"--gpus {world} does not divide the {N_ENVS} environments of the workload")
    n_local = N_ENVS // world

    def env_fn(n):
        return envs.BatchedSyntheticVectorEnv(n, D, A)
    env_fn.vectorized = True

    def make(n_envs, **kw):
        cfg = PPOConfig(num_envs=n_envs, rollout_steps=T, network_hidden_dim=H, num_epochs=E, num_minibatches=MB, verbose=False,
                        total_steps=T * n_envs * 1000, seed=7)
        return PPO(env_fn, cfg, dp=world > 1, dp_exchange=args.dp_exchange, **kw)

    # ---- headline: the ONE 4096 x 128 buffer, env-sharded over the ranks, the reference's global permutation (bit-exact numpy stream) ----
    agent = make(n_local, dp_permutation="global")
    host = synth_host_rollout(1, envs=(rank * n_local, (rank + 1) * n_local))      # this rank's env range of the same global rollout
    buf = RolloutBuffer(ctx, T, n_local, D, 1, False, agent.device)
    buf.load_host(*host)
    torch.cuda.synchronize()
    np.random.seed(123)
    main = time_learn(agent, buf, host, args.steps, args.warmup, world, dist, ctx, keep_outputs=args.dump_outputs is not None and rank == 0)
    agent.engine.check_health()
    if "outputs" in main:
        dump_outputs(args.dump_outputs, main["outputs"])
    ms_per_step, clocks, launches = main["ms"], main["clocks"], main["launches"]
    t_pre, t_gae, t_upd = (main["phases"][k] for k in ("prepass", "gae_and_stats", "update_loop"))
    sample_updates = E * T * N_ENVS
    value = sample_updates / (ms_per_step * 1e-3)
    e2e_value = sample_updates / (main["ms_e2e"] * 1e-3)
    extra = {}
    if world > 1:
        extra["dp_replicas_identical"] = replicas_identical(agent, dist)
        assert extra["dp_replicas_identical"], "data-parallel replicas diverged"
        # the same strong-scaling run with the device permutation generator (no host permutation work; not numpy's numbers)
        ag = make(n_local, dp_permutation="global", minibatch_permutation="device")
        r = time_learn(ag, buf, None, args.steps, args.warmup, world, dist, ctx)
        ag.engine.check_health()
        extra["device_permutation"] = {"value": sample_updates / (r["ms"] * 1e-3), "ms_per_step": r["ms"], "phases_ms": r["phases"],
                                       "replicas_identical": replicas_identical(ag, dist),
                                       "note": "same run with minibatch_permutation='device' (keyed-bijection generator on the GPU)"}
        del ag
        # round 1's measurement: weak scaling, 4096 envs per GPU, rank-local permutations
        if not args.no_weak:
            agw = make(N_ENVS)
            hostw = synth_host_rollout(1 + rank)
            bufw = RolloutBuffer(ctx, T, N_ENVS, D, 1, False, agw.device)
            bufw.load_host(*hostw)
            torch.cuda.synchronize()
            r = time_learn(agw, bufw, None, args.steps, args.warmup, world, dist, ctx)
            extra["weak_scaling"] = {"value": E * T * N_ENVS * world / (r["ms"] * 1e-3), "ms_per_step": r["ms"], "phases_ms": r["phases"],
                                     "envs_per_gpu": N_ENVS, "permutation": "rank-local", "replicas_identical": replicas_identical(agw, dist)}
            del agw, bufw, hostw
            torch.cuda.empty_cache()

    if rank != 0:
        return
    # ---- roofline evidence (rank 0) ----
    fma_peak = bench_fma_peak(ctx)
    gae = bench_gae(ctx, hbm_peak)
    gae_cons = bench_gae(ctx, hbm_peak, settled="rollout")       # only the rollout tensors are promised settled
    gae_plain = bench_gae(ctx, hbm_peak, settled=False)          # no promise, no programmatic dependent launch (the public API's default)
    # a shape where launch latency amortises (SURVEY 8d): 65 536 envs x 128 steps = 235 MB per launch, two buffer sets (470 MB > L2)
    gae_large = bench_gae(ctx, hbm_peak, sets=2, launches=10, settled="rollout", n_envs=65536)
    upd_tflops = E * T * n_local * FLOP_PER_SAMPLE_UPDATE / (t_upd * 1e-3) / 1e12        # per GPU
    # fp32-accurate products cost three TF32 tensor passes; TF32 runs at half the bf16 rate (same cycles per instruction
    # at half the K, confirmed by the in-run probe), so the algorithmic peak is bf16 / 2 / 3
    tensor_peak = bf16_peak / 6.0
    clk_per_mma = bench_mma_probe(ctx)
    sm_mhz = clocks.get("sm_max_mhz") or 1965
    probe_tf32 = 2.0 * 256 * 256 * 8 / clk_per_mma * (ctx.sm_count // 2) * sm_mhz * 1e6 / 1e12
    gemm = bench_dominant_gemm(ctx, tensor_peak)
    peak_note = ("3xTF32 algorithmic peak = MEASURED_PEAKS.json bf16_tflops (%.1f, %s) / 2 (tf32) / 3 (passes); in-run tcgen05 probe: "
                 "%.1f clk per 256x256x8 tf32 MMA = %.0f TF/s tf32 at %d MHz" % (bf16_peak, peak_src, clk_per_mma, probe_tf32, sm_mhz))
    line = {
        "metric": "ppo_update_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(world),
        "phases_ms": {"prepass": t_pre, "gae_and_stats": t_gae, "update_loop": t_upd},
        "update_loop_samples_per_s": E * T * N_ENVS / (t_upd * 1e-3),
        # dominant kernel (52 % of the step in profiles/): algorithmic flops per launch / CUDA-event time of the kernel alone
        "roofline": dict(gemm, peak_source=peak_note, traffic=GEMM_DRAM_TRAFFIC),
        # the whole update loop (32 optimiser steps: gather, forward, loss, backward, reduce, clip + Adam)
        "roofline_update_loop": {"bound": "tensor", "achieved": upd_tflops, "peak": tensor_peak, "unit": "TFLOP/s",
                                 "frac": upd_tflops / tensor_peak, "flop_per_sample_update": FLOP_PER_SAMPLE_UPDATE,
                                 "fp32_fma_peak_tflops": fma_peak, "peak_source": peak_note},
        "roofline_gae": dict(gae, kernel="gae_pipe_kernel (chunked TMA loads, programmatic dependent launch)",
                             peak_source=f"MEASURED_PEAKS.json hbm_gbs ({peak_src})", traffic=GAE_DRAM_TRAFFIC,
                             without_settled_promise={"us_per_launch": gae_cons["us_per_launch"], "achieved": gae_cons["achieved"],
                                                      "frac": gae_cons["frac"], "note": "values / next_values wait for the predecessor grid"},
                             plain_launch_no_promise={"us_per_launch": gae_plain["us_per_launch"], "achieved": gae_plain["achieved"],
                                                      "frac": gae_plain["frac"], "note": "no programmatic dependent launch (calculate_advantage API)"},
                             large_shape_65536x128={"us_per_launch": gae_large["us_per_launch"], "achieved": gae_large["achieved"],
                                                    "frac": gae_large["frac"], "bytes_per_launch": gae_large["bytes_per_launch"],
                                                    "inputs_settled": False}),
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": main["h2d"], "d2h_bytes_per_step": main["d2h"]},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    line.update(extra)
    if world == 1:
        line["train_iteration"] = bench_train_iteration()
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference(3, 1)
        line["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                                "gae_gbps": r["gae_gbps"]}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dp-exchange", default="fused", choices=["fused", "nccl"])
    ap.add_argument("--no-weak", action="store_true", help="skip the extra weak-scaling measurement at --gpus > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed learn() computed (losses, updated parameters) as DIR/<name>.npy; the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
