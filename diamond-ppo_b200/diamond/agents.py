"""PPO and ContinuousPPO agents with the reference's constructor, attributes and methods
(diamond/ppo.py:111-312, diamond/continuous_ppo.py:124-324), running the hot path — rollout
storage, action sampling, pre-update pass, GAE, permutation/gather, MLP forward/backward + loss,
clip + Adam — in libdppo's sm_100a kernels.

Two engines sit behind the same agent API:
  * FusedMlpEngine   — the default networks: every step of learn() is a libdppo kernel over flat
                       parameter buffers (no torch ops, no autograd, no host sync in the loop).
  * AutogradEngine   — a user `network_cls` (readme.md:89-111): the module runs under PyTorch autograd
                       on the GPU; buffer, GAE, gather, loss (+ its gradient) and clip+Adam stay on
                       libdppo kernels.
Env-sharded data parallelism (one process per GPU, torch.distributed/NCCL) is enabled by passing
`process_group=` or by initialising torch.distributed before constructing the agent with `dp=True`.
"""
from __future__ import annotations

import threading
import time
from math import sqrt
from typing import Any, Callable

import numpy as np
import torch
import torch.nn as nn

from . import _native as N
from .config import PPOConfig, ContinuousPPOConfig
from .evaluation import PolicyEvaluation, as_device_obs, select_actions, shared_log_std
from .flat import FlatMlp
from .networks import ActorCriticNetwork, ContinuousActorCriticNetwork, network_parameter_init_
from .utils import Ticker, Logger, Timer, Checkpointer

try:                                    # the real package when present, else the in-repo shim
    import gymnasium as gym             # noqa: F401
except ImportError:                     # pragma: no cover - the GPU image has no gymnasium
    from . import envs as gym


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise N.NativeError("diamond (B200 build) needs a CUDA device: the hot path has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


# ------------------------------------------------------------------------------------------------
# Device-resident rollout buffer (replaces the Python list of NumPy arrays, ppo.py:155-172)
# ------------------------------------------------------------------------------------------------
class RolloutBuffer:
    """Time-major [T, N, ...] device tensors filled one vector step at a time.

    Behaves like the reference's `experience` list (len, iteration, indexing give the six NumPy
    arrays of a step) so user code that inspects `agent.rollout()` keeps working, while
    `agent.learn()` consumes the device tensors directly with no bulk host->device copy."""

    def __init__(self, ctx: N.Context, T: int, N_: int, D: int, A: int, continuous: bool, device: torch.device):
        self.ctx, self.T, self.N, self.D, self.A, self.continuous, self.device = ctx, T, N_, D, A, continuous, device
        f = dict(dtype=torch.float32, device=device)
        self.obs = torch.empty(T, N_, D, **f)
        self.next_obs = torch.empty(T, N_, D, **f)
        self.actions = torch.empty((T, N_, A), **f) if continuous else torch.empty(T, N_, dtype=torch.int32, device=device)
        self.rewards = torch.empty(T, N_, **f)
        self.terminations = torch.empty(T, N_, **f)
        self.truncations = torch.empty(T, N_, **f)
        self.rec_bytes = ctx.step_record_bytes(N_, D, A, continuous)
        padded = (self.rec_bytes + 7) // 8 * 8
        self._pinned = [torch.empty(padded, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self._events = [None, None]
        self._dev_rec = torch.empty(padded, dtype=torch.uint8, device=device)
        self._views = [self._carve(p.numpy()) for p in self._pinned]
        self.h2d_bytes = 0
        self._copy_stream = None        # side stream of load_host
        self._h2d = None                # pending sliced load: {"bounds", "events"}
        self._consumed = None           # event after the last learn() that read this buffer
        self.filled = 0

    def _carve(self, raw: np.ndarray):
        nd = self.N * self.D
        o = 0
        obs = raw[o:o + nd * 4].view(np.float32).reshape(self.N, self.D); o += nd * 4
        nobs = raw[o:o + nd * 4].view(np.float32).reshape(self.N, self.D); o += nd * 4
        rew = raw[o:o + self.N * 8].view(np.float64); o += self.N * 8
        if self.continuous:
            act = raw[o:o + self.N * self.A * 4].view(np.float32).reshape(self.N, self.A); o += self.N * self.A * 4
        else:
            act = raw[o:o + self.N * 8].view(np.int64); o += self.N * 8
        term = raw[o:o + self.N]; o += self.N
        trunc = raw[o:o + self.N]; o += self.N
        assert o == self.rec_bytes
        return obs, nobs, rew, act, term, trunc

    def store(self, t: int, obs, next_obs, actions, rewards, terminations, truncations) -> None:
        """One packed record -> one H2D copy -> one unpack/cast kernel (dppo_buffer_store_step)."""
        slot = t & 1
        if self._events[slot] is not None:
            self._events[slot].synchronize()               # the copy that last read this slot has finished
        v_obs, v_nobs, v_rew, v_act, v_term, v_trunc = self._views[slot]
        np.copyto(v_obs, np.asarray(obs, dtype=np.float32).reshape(self.N, self.D))
        np.copyto(v_nobs, np.asarray(next_obs, dtype=np.float32).reshape(self.N, self.D))
        np.copyto(v_rew, np.asarray(rewards, dtype=np.float64))
        if self.continuous:
            np.copyto(v_act, np.asarray(actions, dtype=np.float32).reshape(self.N, self.A))
        else:
            np.copyto(v_act, np.asarray(actions, dtype=np.int64))
        np.copyto(v_term, np.asarray(terminations, dtype=bool).view(np.uint8))
        np.copyto(v_trunc, np.asarray(truncations, dtype=bool).view(np.uint8))
        self._dev_rec.copy_(self._pinned[slot], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._events[slot] = ev
        self.ctx.buffer_store_step(self._dev_rec, t, self.N, self.D, self.A, self.continuous, self.obs, self.next_obs,
                                   self.actions, self.rewards, self.terminations, self.truncations)
        self.h2d_bytes += self.rec_bytes
        self.filled = max(self.filled, t + 1)

    @classmethod
    def from_lists(cls, ctx, experience, continuous: bool, device) -> "RolloutBuffer":
        """Reference-style experience (list of [obs, next_obs, actions, rewards, term, trunc] NumPy
        arrays, ppo.py:165-172) -> device buffer, with the casts of ppo.py:227-232."""
        obs, nobs, act, rew, term, trunc = (np.asarray(x) for x in zip(*experience))
        T, N_ = rew.shape[:2]
        D = int(np.prod(obs.shape[2:]))
        A = int(np.prod(act.shape[2:])) if continuous else 1
        buf = cls.__new__(cls)
        buf.ctx, buf.T, buf.N, buf.D, buf.A, buf.continuous, buf.device = ctx, T, N_, D, A, continuous, device
        buf._copy_stream, buf._h2d, buf._consumed = None, None, None

        def up(x, dtype):
            t = torch.as_tensor(np.ascontiguousarray(x)).to(dtype)
            return t.pin_memory().to(device, non_blocking=True).contiguous()
        buf.obs = up(obs.reshape(T, N_, D), torch.float32)
        buf.next_obs = up(nobs.reshape(T, N_, D), torch.float32)
        buf.actions = up(act.reshape(T, N_, A), torch.float32) if continuous else up(act, torch.int32)
        buf.rewards, buf.terminations, buf.truncations = up(rew, torch.float32), up(term, torch.float32), up(trunc, torch.float32)
        buf.h2d_bytes = sum(t.numel() * t.element_size() for t in (buf.obs, buf.next_obs, buf.actions, buf.rewards,
                                                                    buf.terminations, buf.truncations))
        buf.filled = T
        return buf

    H2D_CHUNKS = 4

    def load_host(self, obs, next_obs, actions, rewards, terminations, truncations) -> int:
        """Fill the whole buffer from host tensors already in this buffer's dtypes/shapes (pinned memory makes the copies
        asynchronous).  The copies run on a side stream in the order the learner consumes them -- scalars, observations,
        final observations, each observation tensor in H2D_CHUNKS time slices with an event per slice -- so that the
        pre-update pass of slice c overlaps the transfer of slice c+1 (`wait_slice`).  Returns the bytes copied."""
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
        cs = self._copy_stream
        # the old contents may still be read by work already enqueued: wait for the last learn() that consumed THIS buffer when it
        # left a mark (a caller alternating two buffers then overlaps this copy with the other buffer's update loop), else for
        # everything enqueued so far
        if self._consumed is not None:
            cs.wait_event(self._consumed)
        else:
            cs.wait_stream(torch.cuda.current_stream())
        n = 0
        T, nch = self.T, min(self.H2D_CHUNKS, self.T)
        bounds = [T * c // nch for c in range(nch + 1)]
        events = {"obs": [], "next_obs": []}
        with torch.cuda.stream(cs):
            for dst, src in ((self.actions, actions), (self.rewards, rewards), (self.terminations, terminations),
                             (self.truncations, truncations)):
                dst.copy_(src.view(dst.shape), non_blocking=True)
                n += dst.numel() * dst.element_size()
            for name, dst, src in (("obs", self.obs, obs), ("next_obs", self.next_obs, next_obs)):
                src = src.view(dst.shape)
                for c in range(nch):
                    dst[bounds[c]:bounds[c + 1]].copy_(src[bounds[c]:bounds[c + 1]], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record()
                    events[name].append(ev)
                n += dst.numel() * dst.element_size()
        self._h2d = dict(bounds=bounds, events=events)
        self.filled = self.T
        self.h2d_bytes += n
        return n

    def time_slices(self):
        """[(t0, t1)] row ranges in which a pending load_host delivers the observation tensors (one slice otherwise)."""
        if self._h2d is None:
            return [(0, self.T)]
        b = self._h2d["bounds"]
        return [(b[c], b[c + 1]) for c in range(len(b) - 1)]

    def wait_slice(self, name: str, c: int):
        """Makes the current stream wait for slice c of `obs` / `next_obs` of a pending load_host (no-op otherwise)."""
        if self._h2d is not None:
            torch.cuda.current_stream().wait_event(self._h2d["events"][name][c])

    def wait_all(self):
        """Current stream waits for every slice of a pending load_host."""
        if self._h2d is not None:
            for name in ("obs", "next_obs"):
                torch.cuda.current_stream().wait_event(self._h2d["events"][name][-1])
            self._h2d = None

    def h2d_done(self):
        """All slices have been waited for by the consumer: later readers need no further event waits."""
        self._h2d = None

    # ---- list-like view for user code ---------------------------------------------------------
    def __len__(self) -> int:
        return self.filled

    def __getitem__(self, t: int):
        if not -self.filled <= t < self.filled:
            raise IndexError(t)
        self.wait_all()
        act = self.actions[t].cpu().numpy()
        return [self.obs[t].cpu().numpy(), self.next_obs[t].cpu().numpy(),
                act if self.continuous else act.astype(np.int64),
                self.rewards[t].cpu().numpy().astype(np.float64), self.terminations[t].cpu().numpy() != 0,
                self.truncations[t].cpu().numpy() != 0]

    def __iter__(self):
        return (self[t] for t in range(self.filled))


# ------------------------------------------------------------------------------------------------
# Data-parallel plumbing: env-sharded, one process per GPU
# ------------------------------------------------------------------------------------------------
class _Dist:
    """permutation: "local" (default) -- every rank permutes its own shard with its own bit-exact numpy stream and takes
    equal 1/MB slices of it (identical to the reference at one GPU; at G GPUs a valid PPO minibatch scheme that needs no
    host work proportional to the GLOBAL batch); "global" -- every rank generates the reference's permutation of the
    concatenated buffer and keeps its shard's members (sample-for-sample the reference's minibatches, used by the
    equivalence tests; the sequential MT19937 shuffle of G x B indices then runs on every host).
    exchange: "fused" (default on CUDA/NCCL groups) -- dppo_dp_allreduce_clip_adam over NVLink peer memory;
    "nccl" -- torch.distributed all_reduce followed by dppo_clip_adam_step."""

    def __init__(self, group=None, enabled=False, permutation="local", exchange="fused", perm_mode="numpy"):
        import torch.distributed as dist
        self.dist = dist
        self.enabled = bool(enabled or group is not None) and dist.is_available() and dist.is_initialized()
        self.group = group
        self.world = dist.get_world_size(group) if self.enabled else 1
        self.rank = dist.get_rank(group) if self.enabled else 0
        if self.world == 1:
            self.enabled = False
        if permutation not in ("local", "global") or exchange not in ("fused", "nccl") or perm_mode not in ("numpy", "device"):
            raise ValueError("dp_permutation must be 'local' or 'global', dp_exchange 'fused' or 'nccl', "
                             "minibatch_permutation 'numpy' or 'device'")
        self.permutation, self.exchange, self.perm_mode = permutation, exchange, perm_mode
        self.global_perm = self.enabled and permutation == "global"

    def sync_numpy_stream(self, device=None):
        """dp_permutation='global' draws the SAME permutation on every rank from each rank's own numpy global stream: put all
        ranks on rank 0's MT19937 state (a rank whose np.random was consumed differently would otherwise disagree silently on
        minibatch membership; learn() additionally carries a state hash through its all-reduce, FusedMlpEngine.check_health)."""
        if not self.global_perm:
            return
        st = np.random.get_state(legacy=True)
        packed = np.concatenate([np.asarray(st[1], dtype=np.float64), np.array([st[2], st[3], st[4]], dtype=np.float64)])  # exact
        t = torch.as_tensor(packed)
        if self.dist.get_backend(self.group) == "nccl":
            t = t.to(device if device is not None else "cuda")
        src = self.dist.get_global_rank(self.group, 0) if self.group is not None else 0
        self.dist.broadcast(t, src=src, group=self.group)
        packed = t.cpu().numpy()
        np.random.set_state(("MT19937", packed[:624].astype(np.uint32), int(packed[624]), int(packed[625]), float(packed[626])))

    def shared_seed(self, seed, device=None) -> int:
        """The run's base seed for the counter-based generators (action sampling keyed by global env id, device permutation):
        cfg.seed, or a random one when it is None -- in which case rank 0's choice is broadcast so that all ranks agree."""
        if seed is not None:
            return int(seed)
        t = torch.tensor([int.from_bytes(__import__("os").urandom(4), "little") & 0x7FFFFFFF], dtype=torch.int64)
        if self.enabled:
            if self.dist.get_backend(self.group) == "nccl":
                t = t.to(device if device is not None else "cuda")
            src = self.dist.get_global_rank(self.group, 0) if self.group is not None else 0
            self.dist.broadcast(t, src=src, group=self.group)
        return int(t.item())

    def broadcast(self, t: torch.Tensor, src_rank: int):
        if self.enabled:
            src = self.dist.get_global_rank(self.group, src_rank) if self.group is not None else src_rank
            self.dist.broadcast(t, src=src, group=self.group)

    def all_reduce_sum(self, t: torch.Tensor):
        if self.enabled:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)

    def connect_exchange(self, ctx, n_floats, device):
        """Creates this rank's exchange buffer and maps every peer's (CUDA IPC handles all-gathered over the group)."""
        if not self.enabled or self.exchange != "fused" or self.dist.get_backend(self.group) != "nccl":
            return None
        dp = ctx.dp_create(self.world, self.rank, n_floats)
        mine = torch.frombuffer(bytearray(ctx.dp_handle(dp)), dtype=torch.uint8).to(device)
        gathered = [torch.empty_like(mine) for _ in range(self.world)]
        self.dist.all_gather(gathered, mine, group=self.group)
        ctx.dp_connect(dp, b"".join(bytes(g.cpu().numpy().tobytes()) for g in gathered))
        self.dist.barrier(group=self.group)
        return dp


_live_workers: "weakref.WeakSet[_PermWorker]" = None


def _join_workers_at_exit():
    """A speculative worker may still be inside libdppo when the interpreter shuts down: let it finish before its buffers go away."""
    for w in list(_live_workers or ()):
        try:
            w.join(timeout=5.0)
        except RuntimeError:
            pass


class _PermWorker(threading.Thread):
    """Generates the E minibatch permutations of one learn() (ppo.py:252-255) on a host thread while
    the GPU runs the pre-update pass / previous epoch.  Bit-exact continuation of numpy's global
    legacy stream (dppo_permutation_mt19937).  Under data parallelism with the global permutation every rank
    generates the same permutations; the shard filter runs on the device (dppo_perm_shard_filter)."""

    def __init__(self, B_perm, E, MB, outs, owner=None):
        """owner(e) -> bool (optional): under data parallelism with the global permutation the E permutations of a learn() are
        divided among the ranks (epoch e belongs to rank e % world, which broadcasts it over NVLink); a rank only ADVANCES the
        stream over the permutations it does not own (dppo_permutation_mt19937_skip: the draws without the shuffle, ~2.5x
        cheaper), so every rank's stream stays identical while the sequential host work per rank shrinks."""
        super().__init__(daemon=True)
        st = np.random.get_state(legacy=True)
        self.state_tail = (st[3], st[4])
        self.key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
        self.pos = int(st[2])
        # 24-bit hash of the stream state (data-parallel lockstep check: h and h^2 are summed over the ranks in fp64, exactly)
        self.state_hash = float((int(self.key[::7].astype(np.uint64).sum()) * 2654435761 + self.pos * 40503) % (1 << 24))
        self.B, self.E, self.MB, self.outs, self.owner = B_perm, E, MB, outs, owner
        self.start_state = (self.key.copy(), self.pos, self.state_tail)       # what the stream looked like when this worker was created
        self.ready = [threading.Event() for _ in range(E)]
        self.error = None

    def continues(self, B_perm, E, MB) -> bool:
        """True if numpy's global stream is still exactly where this worker started from and the request is the one it was
        started for: a worker started speculatively at the end of the previous learn() (permutations depend on nothing but the
        stream) may then stand in for a fresh one; any np.random use in between invalidates it."""
        st = np.random.get_state(legacy=True)
        key0, pos0, tail0 = self.start_state
        return ((self.B, self.E, self.MB) == (B_perm, E, MB) and st[0] == "MT19937" and int(st[2]) == pos0 and (st[3], st[4]) == tail0
                and np.array_equal(np.asarray(st[1], dtype=np.uint32), key0))

    def run(self):
        try:
            for e in range(self.E):
                if self.owner is None or self.owner(e):
                    _, self.pos = N.permutation_mt19937(self.key, self.pos, self.B, self.outs[e])
                else:
                    self.pos = N.permutation_mt19937_skip(self.key, self.pos, self.B)
                self.ready[e].set()
        except BaseException as ex:      # surfaced by wait()
            self.error = ex
            for ev in self.ready:
                ev.set()

    def start(self):
        """Small batches are permuted inline (a 1024-index permutation takes microseconds; starting and joining a thread ~0.1 ms)."""
        global _live_workers
        self.inline = self.B <= 16384
        if self.inline:
            self.run()
        else:
            if _live_workers is None:
                import atexit
                import weakref
                _live_workers = weakref.WeakSet()
                atexit.register(_join_workers_at_exit)
            _live_workers.add(self)
            super().start()

    def join(self, timeout=None):
        if not getattr(self, "inline", False):
            super().join(timeout)

    def wait(self, e):
        self.ready[e].wait()
        if self.error is not None:
            raise self.error

    def finish(self):
        self.join()
        if self.error is not None:
            raise self.error
        np.random.set_state(("MT19937", self.key, self.pos) + self.state_tail)


def permutation_plan(B: int, world: int, MB: int, global_perm: bool) -> dict:
    """Index space of the minibatch permutation and rows per optimiser step of one rank holding B samples.
    single GPU / DP "local": permutation of this rank's B samples, B/MB rows per step.
    DP "global": ONE permutation of the concatenated buffer on every rank (the reference's, ppo.py:252-255); a rank's share of
    a global minibatch is binomial(M_global, 1/G), so every step runs rows = mean + 6 sigma (rounded up to 128), the index list
    padded with -1: fixed shapes (CUDA-graph replay), padding rows contribute nothing (dppo_perm_shard_filter)."""
    if global_perm and world > 1:
        B_global = B * world
        M_global = B_global // MB
        want = M_global / world + 6.0 * sqrt(M_global * (1.0 / world) * (1.0 - 1.0 / world)) + 16
        rows = min(B, M_global, (int(want) + 127) // 128 * 128)
        return dict(B_perm=B_global, rows=rows, filter=True)
    return dict(B_perm=B, rows=B // MB, filter=False)


# ------------------------------------------------------------------------------------------------
# Engines
# ------------------------------------------------------------------------------------------------
class _EngineBase:
    """State shared by both engines: flat P/G/M/V buffers aliased by the module's parameters."""

    def _adopt(self, network: nn.Module, named_offsets: dict[str, tuple[int, tuple]], total: int):
        dev = self.device
        self.P = torch.zeros(total, dtype=torch.float32, device=dev)
        self.G = torch.zeros(total, dtype=torch.float32, device=dev)
        self.M = torch.zeros(total, dtype=torch.float32, device=dev)
        self.V = torch.zeros(total, dtype=torch.float32, device=dev)
        self.param_list = []
        with torch.no_grad():
            for name, p in network.named_parameters():
                off, shape = named_offsets[name]
                n = p.numel()
                view = self.P[off:off + n].view(*shape)
                view.copy_(p.detach().to(dev, torch.float32).reshape(shape))
                p.data = view                                            # parameters alias the flat buffer
                p.grad = self.G[off:off + n].view(*shape)
                self.param_list.append((name, p, off, n, shape))
        ws_bytes = max(self.ctx.clip_adam_workspace_bytes(total), self.ctx.dp_workspace_bytes(total))
        self.adam_ws = torch.empty(ws_bytes // 8 + 1, dtype=torch.float64, device=dev)
        self.grad_norm = torch.zeros(1, dtype=torch.float32, device=dev)
        self.total = total
        self.dpx = None
        self.grad_sumsq = torch.zeros(self.ctx.grad_sumsq_bytes(total) // 8 + 1, dtype=torch.float64, device=dev)
        self.adam_step = 0

    def bind_optimizer(self, optimizer: torch.optim.Optimizer):
        """Expose the kernel-side Adam moments through optimizer.state so `optimizer.state_dict()`
        (Checkpointer, utils.py:584-600) reflects them."""
        self.optimizer = optimizer
        for name, p, off, n, shape in self.param_list:
            optimizer.state[p] = {"step": torch.tensor(float(self.adam_step)),
                                  "exp_avg": self.M[off:off + n].view(*shape),
                                  "exp_avg_sq": self.V[off:off + n].view(*shape)}
        optimizer._opt_called = True      # the kernels are the optimiser step; silences LinearLR's ordering warning

    def _resync_optimizer(self):
        """If user code replaced optimizer state / parameter storage (load_state_dict), pull it back
        into the flat buffers and re-alias."""
        for name, p, off, n, shape in self.param_list:
            if p.data_ptr() != self.P[off:off + n].data_ptr():
                self.P[off:off + n].view(*shape).copy_(p.detach())
                p.data = self.P[off:off + n].view(*shape)
            if p.grad is None or p.grad.data_ptr() != self.G[off:off + n].data_ptr():
                p.grad = self.G[off:off + n].view(*shape)
            st = self.optimizer.state.get(p)
            if st and st["exp_avg"].data_ptr() != self.M[off:off + n].data_ptr():
                self.M[off:off + n].view(*shape).copy_(st["exp_avg"])
                self.V[off:off + n].view(*shape).copy_(st["exp_avg_sq"])
                self.adam_step = int(float(st["step"]))
                st["exp_avg"], st["exp_avg_sq"] = self.M[off:off + n].view(*shape), self.V[off:off + n].view(*shape)

    def _publish_steps(self):
        for _, p, *_ in self.param_list:
            self.optimizer.state[p]["step"] = torch.tensor(float(self.adam_step))

    def _hyper(self, cfg, M_global, B_global) -> N.Hyper:
        h = N.Hyper()
        h.ppo_clip, h.value_loss_weight, h.entropy_beta = cfg.ppo_clip, cfg.value_loss_weight, cfg.entropy_beta
        h.grad_norm_clip, h.adam_eps = cfg.grad_norm_clip, cfg.adam_eps
        h.beta1, h.beta2 = self.optimizer.param_groups[0]["betas"]
        h.lr = self.optimizer.param_groups[0]["lr"]
        h.advantage_norm, h.adv_count, h.loss_denominator = int(cfg.advantage_norm), B_global, M_global
        return h


class FusedMlpEngine(_EngineBase):
    """learn() for the default MLP networks: libdppo kernels only."""

    fused = True

    def __init__(self, ctx, network, cfg, obs_dim, act_dim, continuous, device, dist: _Dist):
        self.ctx, self.cfg, self.device, self.dist, self.continuous = ctx, cfg, device, dist, continuous
        self.network = network
        self.fm = FlatMlp(obs_dim, cfg.network_hidden_dim, act_dim, continuous)
        self._adopt(network, self.fm.slices, self.fm.total)
        self.dpx = dist.connect_exchange(ctx, self.fm.total, device)    # fused NVLink exchange (None: single GPU / NCCL path)
        self.D, self.A = obs_dim, act_dim
        self.fwd_rows = 65536
        self.speculate_permutations = True      # generate the next learn()'s numpy-stream permutations in the background (validated)
        self.fwd_ws = torch.empty(ctx.mlp_workspace_bytes(self.fm.desc, self.fwd_rows, False) // 4 + 256, device=device)
        # heads of the training step: the fused head kernel where it takes the shape (A <= 32 and (A+1) H within its shared
        # memory), else GEMM heads (hidden <= 2048, up to 1024 actions); both write the same flat gradient and losses
        self.fused_heads = ctx.mlp_fused_heads_supported(self.fm.desc)
        if self.fused_heads:
            self._grad_minibatch, self._train_ws_bytes = ctx.mlp_grad_minibatch, (lambda rows: ctx.mlp_workspace_bytes(self.fm.desc, rows, True))
        else:
            self._grad_minibatch, self._train_ws_bytes = ctx.mlp_grad_minibatch_gemm_heads, (lambda rows: ctx.mlp_gemm_heads_workspace_bytes(self.fm.desc, rows))
        self._train_ws = None
        self._bufs = {}
        self.draws = 0
        self.seed = dist.shared_seed(cfg.seed, device)
        self._act_stage = {}
        self.last_losses = None
        self.timing = {}
        self.use_graphs = True          # replay the optimiser steps of an epoch as a CUDA graph (single GPU, steady state)
        self._seen_keys = []
        self.reuse_rollout_values = True   # learn() takes log-probs / values recorded at sampling time when they are still valid
        self.use_small_kernel = True       # default 64-wide nets: the whole update loop of a learn() as one cluster launch
        self.dp_seq = 0                    # data-parallel exchanges issued so far (monotonic; independent of the Adam step)
        self.perm_mode = dist.perm_mode    # "numpy": bit-exact np.random stream on a host thread; "device": keyed-bijection generator
        self.perm_seed = (self.seed * 0x9E3779B97F4A7C15 + (0 if dist.global_perm or not dist.enabled else dist.rank + 1)) % (1 << 64)
        self.perm_counter = 0
        self._pending_check = None

    # ---- rollout side: fused forward + sampling (ppo.py:73-82) -----------------------------------
    def sample_actions(self, observations: np.ndarray) -> np.ndarray:
        n = observations.shape[0]
        st = self._act_stage.get(n)
        if st is None:
            st = dict(h_obs=torch.empty(n, self.D, dtype=torch.float32).pin_memory(),
                      d_obs=torch.empty(n, self.D, dtype=torch.float32, device=self.device),
                      head=torch.empty(n, self.A, dtype=torch.float32, device=self.device),
                      d_act=(torch.empty(n, self.A, dtype=torch.float32, device=self.device) if self.continuous
                             else torch.empty(n, dtype=torch.int64, device=self.device)))
            st["h_act"] = torch.empty(st["d_act"].shape, dtype=st["d_act"].dtype).pin_memory()
            self._act_stage[n] = st
        np.copyto(st["h_obs"].numpy(), np.asarray(observations, dtype=np.float32).reshape(n, self.D))
        st["d_obs"].copy_(st["h_obs"], non_blocking=True)
        self.ctx.mlp_forward(self.fm.desc, self.P, st["d_obs"], n, 1, st["head"], None, self.fwd_ws)
        env_offset = self.dist.rank * n
        if self.continuous:
            lay = self.fm.layout
            self.ctx.sample_gaussian(st["head"], self.P[lay.log_std:lay.log_std + self.A], self.seed, self.draws, env_offset, st["d_act"])
        else:
            self.ctx.sample_categorical(st["head"], self.seed, self.draws, env_offset, st["d_act"])
        self.draws += 1
        st["h_act"].copy_(st["d_act"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return st["h_act"].numpy().copy()

    def sample_actions_device(self, d_obs: torch.Tensor, values_out: torch.Tensor | None = None,
                              logp_out: torch.Tensor | None = None, counter: int | None = None) -> torch.Tensor:
        """get_actions for observations that already live on the device (DeviceVectorEnv): forward + sampling kernels only,
        no host round trip and no synchronisation.  Returns int64 [N] / f32 [N, A] on the device.  values_out / logp_out
        (f32 [N]) additionally receive V(obs) and log_prob(action) of the sampling policy (SURVEY.md 8f-2)."""
        n = d_obs.shape[0]
        st = self._act_stage.get(("dev", n))
        if st is None:
            st = dict(head=torch.empty(n, self.A, dtype=torch.float32, device=self.device),
                      d_act=(torch.empty(n, self.A, dtype=torch.float32, device=self.device) if self.continuous
                             else torch.empty(n, dtype=torch.int64, device=self.device)))
            self._act_stage[("dev", n)] = st
        self.ctx.mlp_forward(self.fm.desc, self.P, d_obs, n, 1 if values_out is None else 3, st["head"], values_out, self.fwd_ws)
        env_offset = self.dist.rank * n
        draw = self.draws if counter is None else counter      # counter: relative draw index of a captured rollout (see _PPOBase.rollout)
        if self.continuous:
            lay = self.fm.layout
            self.ctx.sample_gaussian(st["head"], self.P[lay.log_std:lay.log_std + self.A], self.seed, draw, env_offset, st["d_act"],
                                     logp_out)
        else:
            self.ctx.sample_categorical(st["head"], self.seed, draw, env_offset, st["d_act"], logp_out)
        if counter is None:
            self.draws += 1
        return st["d_act"]

    def policy_stamp(self):
        """Identifies the parameter values: optimiser steps taken by the kernels + torch-side in-place writes to the flat buffer."""
        return (self.adam_step, self.P._version, self.P.data_ptr(), sum(p._version for _, p, *_ in self.param_list))

    # ---- learn (ppo.py:224-287) ---------------------------------------------------------------------
    def _plan(self, T, N_, MB):
        return permutation_plan(T * N_, self.dist.world if self.dist.enabled else 1, MB, self.dist.global_perm)

    def _alloc(self, T, N_, E, MB):
        key = (T, N_, E, MB, self.dist.global_perm)
        if key in self._bufs:
            return self._bufs[key]
        dev, B = self.device, T * N_
        plan = self._plan(T, N_, MB)
        f = dict(dtype=torch.float32, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        b = dict(head=torch.empty(B, self.A, **f), values=torch.empty(T, N_, **f), next_values=torch.empty(T, N_, **f),
                 old_logp=torch.empty(T, N_, **f), adv=torch.empty(T, N_, **f), ret=torch.empty(T, N_, **f),
                 stats=torch.zeros(4, dtype=torch.float64, device=dev), losses=torch.zeros(E * MB, 4, **f),
                 # per-epoch staging, double-buffered by epoch parity: the step indices [MB * rows] and, when they are derived on
                 # the device (shard filter), the permutation they are derived from
                 idx=[torch.empty(MB * plan["rows"], **i32) for _ in range(2)],
                 perm=[torch.empty(plan["B_perm"], **i32) for _ in range(2)] if plan["filter"] else None,
                 counts=[torch.zeros(MB, **i32) for _ in range(2)], overflow=torch.zeros(1, **i32),
                 # pinned staging of the host permutations: two sets, alternating between consecutive learn() calls, so that the host
                 # worker of learn k+1 never waits for the last asynchronous copy of learn k
                 h_sets=[[torch.empty(plan["B_perm"], dtype=torch.int32).pin_memory() for _ in range(E)] for _ in range(2)],
                 h_set=0, h_consumed=[None, None],
                 copy_stream=torch.cuda.Stream(), copied=[torch.cuda.Event() for _ in range(2)],
                 done=[torch.cuda.Event() for _ in range(2)], plan=plan)
        for ev in b["done"]:
            ev.record()
        b["train_ws"] = torch.empty(self._train_ws_bytes(plan["rows"]) // 4 + 256, **f)
        b["m_max"] = plan["rows"]
        self._bufs[key] = b
        return b

    def _stage_epoch(self, b, worker, e, T, N_, MB):
        """Fills b["idx"][e & 1] with the MB index lists of epoch e ON THE SIDE STREAM and records b["copied"][e & 1]: bit-exact numpy
        stream (host worker -> pinned buffer -> async copy; under the DP global permutation generated by rank e mod G only and broadcast
        over NVLink) or the device generator, then -- DP "global" -- the shard filter.  Callers stage epoch e + 1 right after they have
        enqueued epoch e, so host shuffle, copy, broadcast and filter all run under the previous epoch's optimiser steps; the
        consumer waits for the event with `_await_epoch`."""
        p = e & 1
        plan, ctx, dist = b["plan"], self.ctx, self.dist
        target = b["perm"][p] if plan["filter"] else b["idx"][p]
        cs = b["copy_stream"]
        owner = (e % dist.world) if plan["filter"] else dist.rank              # global permutation: epoch e is generated by one rank
        if worker is not None and owner == dist.rank:
            worker.wait(e)
        cs.wait_event(b["done"][p])                                      # the steps that last read idx[p] / perm[p] have finished
        with torch.cuda.stream(cs):
            if worker is not None:
                if owner == dist.rank:
                    target.copy_(b["h_idx"][e], non_blocking=True)
                    b["h_consumed"][b["h_set"]] = torch.cuda.Event()
                    b["h_consumed"][b["h_set"]].record()
                if plan["filter"]:
                    dist.broadcast(target, owner)                        # 4 bytes per index over NVLink instead of a shuffle per rank
            else:
                ctx.permutation_device(self.perm_seed, self.perm_counter, plan["B_perm"], target)
                self.perm_counter += 1
            if plan["filter"]:
                ctx.perm_shard_filter(b["perm"][p], plan["B_perm"], N_ * dist.world, dist.rank * N_, N_, MB, plan["rows"], b["idx"][p],
                                      b["counts"][p], b["overflow"])
            b["copied"][p].record()

    def _await_epoch(self, b, e):
        torch.cuda.current_stream().wait_event(b["copied"][e & 1])
        return b["idx"][e & 1]

    SMALL_ROWS = 1024      # minibatch rows up to which the one-launch cluster kernel beats the per-layer kernels

    def _learn_small(self, b, worker, hyper, desc, tensors, losses, E, MB, rows):
        """Default 64-wide networks: all E x MB optimiser steps in ONE launch (dppo_small_update) -- parameters, gradient partials
        and sharded Adam state live in the distributed shared memory of an 8-CTA cluster for the whole update loop."""
        ctx, dev = self.ctx, self.device
        S, B = E * MB, MB * rows
        sm = b.get("small")
        if sm is None:
            sm = b["small"] = dict(idx=torch.empty(E * B, dtype=torch.int32, device=dev), consts=torch.empty(S, 2, dtype=torch.float32, device=dev),
                                   h_consts=torch.empty(S, 2, dtype=torch.float32).pin_memory(), copied=None)
        if sm["copied"] is not None:
            sm["copied"].synchronize()                                   # the previous copy out of h_consts has completed
        hc = sm["h_consts"].numpy()
        b1, b2 = hyper.beta1, hyper.beta2
        for k in range(S):
            step = self.adam_step + k + 1                                # torch/optim/adam.py:531-547, python-float bias corrections
            hc[k, 0] = np.float32(np.sqrt(1.0 - b2 ** step))
            hc[k, 1] = np.float32(-(hyper.lr / (1.0 - b1 ** step)))
        sm["consts"].copy_(sm["h_consts"], non_blocking=True)
        sm["copied"] = torch.cuda.Event()
        sm["copied"].record()
        for e in range(E):
            if worker is not None:
                worker.wait(e)
                sm["idx"][e * B:(e + 1) * B].copy_(b["h_idx"][e], non_blocking=True)
                b["h_consumed"][b["h_set"]] = torch.cuda.Event()
                b["h_consumed"][b["h_set"]].record()
            else:
                ctx.permutation_device(self.perm_seed, self.perm_counter, B, sm["idx"][e * B:(e + 1) * B])
                self.perm_counter += 1
        hyper.step = self.adam_step + 1
        obs_flat, actions, old_logp, adv, ret = tensors
        ctx.small_update(desc, self.P, self.G, self.M, self.V, obs_flat, actions, old_logp, adv, ret, b["stats"], sm["idx"], rows, S, hyper,
                         sm["consts"], losses, self.grad_norm)
        self.adam_step += S

    def _step(self, b, hyper, desc, tensors, idx_k, rows, losses_k, seq):
        """One optimiser step on the current stream: minibatch gradient, [exchange,] clip + Adam."""
        ctx = self.ctx
        obs_flat, actions, old_logp, adv, ret = tensors
        if self.dpx is not None:
            # env-sharded DP, fused exchange: the local gradient and loss sums go straight into this exchange's slot of the
            # exchange buffer; one kernel per rank then sums all ranks' slots over NVLink and starts the optimiser step
            slot = ctx.dp_slot(self.dpx, seq)
            self._grad_minibatch(desc, self.P, slot, obs_flat, actions, old_logp, adv, ret, b["stats"], idx_k, rows, hyper,
                                 slot + 4 * self.total, b["train_ws"])
            ctx.dp_allreduce_clip_adam(self.dpx, seq, self.P, self.G, self.M, self.V, hyper, losses_k, self.adam_ws, self.grad_norm)
            return
        self._grad_minibatch(desc, self.P, self.G, obs_flat, actions, old_logp, adv, ret, b["stats"], idx_k, rows, hyper, losses_k,
                             b["train_ws"])
        if self.dist.enabled:
            self.dist.all_reduce_sum(self.G)              # env-sharded DP over NCCL: sum of per-shard gradients
            self.dist.all_reduce_sum(losses_k)
        ctx.clip_adam_step(self.P, self.G, self.M, self.V, hyper, self.adam_ws, self.grad_norm)

    def _learn_epochs_graphed(self, b, worker, hyper, desc, tensors, losses, E, MB, T, N_, key):
        """The MB optimiser steps of an epoch replayed as ONE CUDA graph.  Everything that changes between replays is
        device-resident: the step indices (b["idx"][parity], refilled per epoch), Adam's two step-dependent constants and, under
        data parallelism, the exchange sequence number."""
        ctx, dev = self.ctx, self.device
        rows = b["plan"]["rows"]
        graphs = b.setdefault("graph", {})                               # one captured pair per set of baked-in pointers
        gs = graphs.get(key)
        if gs is None:
            if len(graphs) >= 4:                                         # bounded: callers cycling through many buffers re-capture
                graphs.pop(next(iter(graphs)))
            gs = dict(key=key, graphs=[], launches=0,
                      consts=[torch.zeros(MB, 4, dtype=torch.float32, device=dev) for _ in range(2)],
                      h_consts=[torch.zeros(MB, 4, dtype=torch.float32).pin_memory() for _ in range(2)],
                      losses=[torch.zeros(MB, 4, dtype=torch.float32, device=dev) for _ in range(2)],
                      consts_copied=[torch.cuda.Event() for _ in range(2)])
            cap = torch.cuda.Stream()
            cap.wait_stream(torch.cuda.current_stream())
            for p in range(2):
                g = torch.cuda.CUDAGraph()
                l0 = ctx.launches
                with torch.cuda.graph(g, stream=cap):
                    for k in range(MB):
                        # Adam's constants and the exchange sequence number are read from consts[p][k]; only the PARITY of the
                        # sequence number is baked in (exchange slot): replays start on an odd sequence number (dp_seq even)
                        hyper.step = 1
                        hyper.step_consts = gs["consts"][p][k].data_ptr()
                        self._step(b, hyper, desc, tensors, b["idx"][p][k * rows:(k + 1) * rows], rows, gs["losses"][p][k], k + 1)
                gs["launches"] = ctx.launches - l0
                gs["graphs"].append(g)
            hyper.step_consts = None
            torch.cuda.current_stream().wait_stream(cap)
            graphs[key] = gs
        main = torch.cuda.current_stream()
        b1, b2 = hyper.beta1, hyper.beta2
        self._stage_epoch(b, worker, 0, T, N_, MB)
        for e in range(E):
            p = e & 1
            gs["consts_copied"][p].synchronize()                         # the previous copy out of h_consts[p] is done
            hc = gs["h_consts"][p].numpy()
            hc_seq = hc.view(np.uint64)                                  # [MB, 2]: column 1 aliases floats 2..3
            for k in range(MB):
                step = self.adam_step + k + 1                            # torch/optim/adam.py:531-547, python-float bias corrections
                hc[k, 0] = np.float32(np.sqrt(1.0 - b2 ** step))
                hc[k, 1] = np.float32(-(hyper.lr / (1.0 - b1 ** step)))
                hc_seq[k, 1] = self.dp_seq + k + 1
            self._await_epoch(b, e)
            gs["consts"][p].copy_(gs["h_consts"][p], non_blocking=True)  # stream-ordered after the graph that last read consts[p]
            gs["consts_copied"][p].record()
            gs["graphs"][p].replay()
            losses[e * MB:(e + 1) * MB].copy_(gs["losses"][p])
            b["done"][p].record()
            if e + 1 < E:
                self._stage_epoch(b, worker, e + 1, T, N_, MB)            # under this epoch's optimiser steps
            self.adam_step += MB
            self.dp_seq += MB
            ctx.count_launches(gs["launches"])

    def prepass(self, buf: RolloutBuffer, b):
        """ppo.py:235-238: old log-probs, values, next_values with the pre-update parameters."""
        B = buf.T * buf.N
        N_ = buf.N
        ctx, desc = self.ctx, self.fm.desc
        # time slices: one for a resident buffer; a pending load_host delivers the observations slice by slice and the
        # forward pass of slice c overlaps the transfer of slice c+1
        slices = buf.time_slices()
        values, next_values = b["values"].view(B), b["next_values"].view(B)
        for c, (t0, t1) in enumerate(slices):
            buf.wait_slice("obs", c)
            r0, r1 = t0 * N_, t1 * N_
            ctx.mlp_forward(desc, self.P, buf.obs[t0:t1], r1 - r0, 3, b["head"][r0:r1], values[r0:r1], self.fwd_ws)
        if self.continuous:
            lay = self.fm.layout
            ctx.logprob_gaussian(b["head"], self.P[lay.log_std:lay.log_std + self.A], buf.actions.view(B, self.A), b["old_logp"].view(B))
        else:
            ctx.logprob_categorical(b["head"], buf.actions.view(B), b["old_logp"].view(B))
        for c, (t0, t1) in enumerate(slices):
            buf.wait_slice("next_obs", c)
            r0, r1 = t0 * N_, t1 * N_
            ctx.mlp_forward(desc, self.P, buf.next_obs[t0:t1], r1 - r0, 2, None, next_values[r0:r1], self.fwd_ws)
        buf.h2d_done()

    def prepass_from_rollout(self, buf: RolloutBuffer, b):
        """SURVEY.md 8f-2: the pre-update pass (ppo.py:235-238) re-evaluates the policy that sampled the rollout, with unchanged
        parameters.  When the rollout recorded log_prob(action) and V(obs) at sampling time, only V(final observation) is
        missing, and `next_obs[t] == obs[t+1]` wherever the environment did not finish at t: next_values[t] = values[t+1]
        there, and the critic is evaluated only on the final observations of finished steps and on the last row --
        ~3 % of the 2 B rows the full pass touches."""
        T, N_ = buf.T, buf.N
        b["values"].copy_(buf.values)
        b["old_logp"].copy_(buf.logp)
        ws = b.get("next_ws")
        if ws is None:
            ws = b["next_ws"] = torch.empty(self.ctx.mlp_next_values_workspace_bytes(self.fm.desc, T, N_), dtype=torch.uint8, device=self.device)
        # row selection, gather, critic and scatter all take their row count from device memory: no host synchronisation
        self.ctx.mlp_next_values(self.fm.desc, self.P, buf.next_obs.view(T * N_, self.D), buf.terminations, buf.truncations, buf.values,
                                 b["next_values"], ws)

    def check_health(self):
        """Raises if an earlier learn() detected (asynchronously) a data-parallel fault: ranks whose numpy permutation streams
        disagree, a shard-filter overflow, or an exchange kernel that timed out waiting for a peer.  Called at the start of every
        learn() and by train() at its end; costs no device synchronisation."""
        if self.dpx is not None:
            st = self.ctx.dp_status(self.dpx)
            if st != 0:
                raise N.NativeError(f"data-parallel exchange timed out waiting for rank {st - 1} (crashed or desynchronised peer)")
        chk = self._pending_check
        if chk is not None and chk["event"].query():
            self._pending_check = None
            s1, s2, over = (float(x) for x in chk["host"])
            if over != 0:
                raise RuntimeError("dp_permutation='global': a rank's share of a global minibatch exceeded the padded step size "
                                   "(6-sigma bound); the update of that learn() dropped samples")
            if abs(s2 * self.dist.world - s1 * s1) > 0.5:
                raise RuntimeError("dp_permutation='global': the ranks' numpy permutation streams disagree (np.random was consumed "
                                   "differently per rank); minibatch membership is inconsistent")

    def learn(self, buf: RolloutBuffer, events=None):
        cfg, ctx, dist = self.cfg, self.ctx, self.dist
        T, N_ = buf.T, buf.N
        E, MB = cfg.num_epochs, cfg.num_minibatches
        B = T * N_
        B_global = B * dist.world
        if B_global % MB != 0:              # the reference's reshape raises here (ppo.py:255)
            raise ValueError(f"cannot reshape array of size {E * B_global} into shape ({E},{MB},{B_global // MB})")
        M_global = B_global // MB
        self.check_health()
        self._resync_optimizer()
        b = self._alloc(T, N_, E, MB)
        plan = b["plan"]
        if plan["B_perm"] % MB != 0:
            raise ValueError(f"cannot reshape array of size {E * plan['B_perm']} into shape ({E},{MB},{plan['B_perm'] // MB})")
        worker = None
        lock_hash = 0.0
        b["h_set"] ^= 1                      # host-side staging buffers alternate between consecutive learn() calls
        if self.perm_mode == "numpy":
            b["h_idx"] = b["h_sets"][b["h_set"]]
            owner = (lambda e: e % dist.world == dist.rank) if plan["filter"] else None
            spec = b.pop("spec", None)
            if spec is not None and spec.continues(plan["B_perm"], E, MB):
                worker = spec                   # started at the end of the previous learn(): the permutations are (being) generated already
            else:
                if spec is not None:
                    spec.join()                 # the stream moved on (np.random was used in between): its permutations are discarded
                if b["h_consumed"][b["h_set"]] is not None:
                    b["h_consumed"][b["h_set"]].synchronize()   # the async copies out of this pinned set (two learn() calls ago) are done
                worker = _PermWorker(plan["B_perm"], E, MB, [h.numpy() for h in b["h_idx"]], owner)
                worker.start()                  # host permutation overlaps the pre-update pass on the GPU
            lock_hash = worker.state_hash

        def mark(name):
            if events is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                events[name] = ev
        mark("start")
        if self.reuse_rollout_values and getattr(buf, "policy_stamp", None) == self.policy_stamp():
            self.prepass_from_rollout(buf, b)
        else:
            self.prepass(buf, b)
        mark("prepass_end")
        b["stats"].zero_()
        if dist.global_perm:                # ranks must hold the same numpy stream: 24-bit state hash h and h^2 ride in the all-reduce
            lk = b.setdefault("lock_host", [torch.zeros(2, dtype=torch.float64).pin_memory() for _ in range(2)])[b["h_set"]]
            lk[0], lk[1] = lock_hash, lock_hash * lock_hash            # pinned: the copy below must not block the host on the stream
            b["stats"][2:4].copy_(lk, non_blocking=True)
        # the kernel right before the GAE launch is a 32-byte fill, not the pre-update pass: inputs are settled
        ctx.gae(buf.rewards, buf.terminations, buf.truncations, b["values"], b["next_values"], cfg.gamma, cfg.gae_lambda,
                advantages=b["adv"], returns=b["ret"], stats=b["stats"], inputs_settled=True)
        dist.all_reduce_sum(b["stats"])     # global mean/std of the advantages (ppo.py:243)
        mark("gae_end")

        hyper = self._hyper(cfg, M_global, B_global)
        desc = self.fm.desc
        tensors = (buf.obs.view(B, self.D), buf.actions.view(B, self.A) if self.continuous else buf.actions.view(B),
                   b["old_logp"].view(B), b["adv"].view(B), b["ret"].view(B))
        losses = b["losses"]
        rows = plan["rows"]
        # Steady state: the MB optimiser steps of an epoch are replayed as one CUDA graph (kernel-to-kernel launch gaps are 6 % of
        # the step otherwise, far more at data-parallel step sizes).  The graph is keyed on the data pointers it bakes in and
        # only used from the second consecutive learn() on the same buffers.
        ptr_key = (buf.obs.data_ptr(), buf.actions.data_ptr(), buf.T, buf.N, E, MB, cfg.ppo_clip, cfg.value_loss_weight,
                   cfg.entropy_beta, cfg.grad_norm_clip, cfg.adam_eps, bool(cfg.advantage_norm), dist.global_perm)
        # under DP: fused exchange only, and an even MB so that the baked slot parity repeats
        dp_ok = not dist.enabled or (self.dpx is not None and MB % 2 == 0 and self.dp_seq % 2 == 0)
        # (double-buffered callers alternate between two rollout buffers: both keys are remembered)
        use_graph = self.use_graphs and dp_ok and ptr_key in self._seen_keys
        self._seen_keys = (self._seen_keys + [ptr_key])[-4:] if ptr_key not in self._seen_keys else self._seen_keys
        if not dist.enabled:
            hyper.grad_sumsq = self.grad_sumsq.data_ptr()    # gradient assembly leaves the norm partials for the Adam kernel
        if self.use_small_kernel and not dist.enabled and rows <= self.SMALL_ROWS and ctx.small_update_supported(desc):
            self._learn_small(b, worker, hyper, desc, tensors, losses, E, MB, rows)
        elif use_graph:
            self._learn_epochs_graphed(b, worker, hyper, desc, tensors, losses, E, MB, T, N_, ptr_key)
        else:
            self._stage_epoch(b, worker, 0, T, N_, MB)
            for e in range(E):
                idx = self._await_epoch(b, e)
                for k in range(MB):
                    self.adam_step += 1
                    self.dp_seq += 1
                    hyper.step = self.adam_step
                    self._step(b, hyper, desc, tensors, idx[k * rows:(k + 1) * rows], rows, losses[e * MB + k], self.dp_seq)
                b["done"][e & 1].record()
                if e + 1 < E:
                    self._stage_epoch(b, worker, e + 1, T, N_, MB)        # under this epoch's optimiser steps
        mark("update_end")
        if dist.global_perm:                 # verified lazily by check_health(): no synchronisation here
            host = b.setdefault("check_host", [torch.zeros(3, dtype=torch.float64).pin_memory() for _ in range(2)])[b["h_set"]]
            host.copy_(torch.cat([b["stats"][2:4], b["overflow"].double()]), non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            self._pending_check = dict(host=host, event=ev)
        if worker is not None:
            worker.finish()
            if self.speculate_permutations and not worker.inline:
                # The next learn()'s permutations depend on nothing but numpy's stream, which now stands where that learn() will find
                # it: generate them in the background already (into the other pinned set).  At data-parallel step sizes an epoch
                # of optimiser steps is shorter than one 524 288-index MT19937 shuffle, so a worker started inside learn() leaves the
                # GPU waiting; a worker started one learn() ahead does not.  Adopted only if the stream is untouched (continues()).
                nxt = b["h_set"] ^ 1
                if b["h_consumed"][nxt] is not None:
                    b["h_consumed"][nxt].synchronize()
                owner = (lambda e: e % dist.world == dist.rank) if plan["filter"] else None
                b["spec"] = _PermWorker(plan["B_perm"], E, MB, [h.numpy() for h in b["h_sets"][nxt]], owner)
                b["spec"].start()
        self._publish_steps()
        self.last_losses = losses
        buf._consumed = torch.cuda.Event()
        buf._consumed.record()


class AutogradEngine(_EngineBase):
    """learn() for a user network_cls: module under torch autograd, everything else on libdppo kernels."""

    def __init__(self, ctx, network, cfg, continuous, device, dist: _Dist):
        self.ctx, self.cfg, self.device, self.dist, self.continuous = ctx, cfg, device, dist, continuous
        self.network = network
        offsets, o = {}, 0
        for name, p in network.named_parameters():
            offsets[name] = (o, tuple(p.shape))
            o += (p.numel() + 3) // 4 * 4
        self._adopt(network, offsets, max(o, 4))
        self.last_losses = None

    def learn(self, buf: RolloutBuffer, events=None):
        cfg, ctx, dist, net = self.cfg, self.ctx, self.dist, self.network
        # Env-sharded data parallelism for a user module: rank-local permutations (equal 1/MB slices of every shard), loss means over the
        # GLOBAL minibatch, gradients and loss sums summed over the ranks with NCCL before the clip (ppo.py:284); the advantage
        # statistics are global too.  (The fused NVLink exchange needs the flat-gradient kernels of the default networks.)
        T, N_ = buf.T, buf.N
        E, MB = cfg.num_epochs, cfg.num_minibatches
        B = T * N_
        if B % MB != 0:
            raise ValueError(f"cannot reshape array of size {E * B} into shape ({E},{MB},{B // MB})")
        M = B // MB
        self._resync_optimizer()
        dev = self.device
        h_idx = [torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(E)]
        worker = _PermWorker(B, E, MB, [h.numpy() for h in h_idx])
        worker.start()
        buf.wait_all()
        obs, nobs = buf.obs, buf.next_obs
        A = buf.A
        old_logp = torch.empty(B, device=dev)
        with torch.inference_mode():
            if self.continuous:
                means, log_stds, values = net.get_means_log_stds_and_values(obs)
                ls = log_stds.reshape(B, A)
                if bool((ls == ls[:1]).all()):                         # state-independent std: shared [A] vector
                    ctx.logprob_gaussian(means.reshape(B, A).contiguous(), ls[0].contiguous(), buf.actions.view(B, A), old_logp)
                else:
                    old_logp.copy_(torch.distributions.Normal(means, log_stds.exp()).log_prob(buf.actions).sum(-1).reshape(B))
            else:
                logits, values = net.get_logits_and_values(obs)
                ctx.logprob_categorical(logits.reshape(B, -1).contiguous(), buf.actions.view(B), old_logp)
                n_out = logits.shape[-1]                               # the buffer keeps one action index per sample
            next_values = net.get_values(nobs)
        values = values.reshape(T, N_).contiguous().clone()
        next_values = next_values.reshape(T, N_).contiguous().clone()
        stats = torch.zeros(2, dtype=torch.float64, device=dev)
        adv = torch.empty(T, N_, device=dev)
        ret = torch.empty(T, N_, device=dev)
        ctx.gae(buf.rewards, buf.terminations, buf.truncations, values, next_values, cfg.gamma, cfg.gae_lambda,
                advantages=adv, returns=ret, stats=stats)
        dist.all_reduce_sum(stats)                     # global mean / std of the advantages (ppo.py:243)
        if cfg.advantage_norm:
            adv = ctx.adv_normalize(adv, stats, B * dist.world)
        hyper = self._hyper(cfg, M * dist.world, B * dist.world)
        hyper.advantage_norm = 0                       # already normalised above
        obs_flat, adv_f, ret_f = obs.view(B, -1), adv.view(B), ret.view(B)
        act_bits = buf.actions.view(B, A) if self.continuous else buf.actions.view(B).view(torch.float32)
        losses = torch.zeros(E * MB, 4, device=dev)
        loss_ws = torch.empty(ctx.ppo_loss_workspace_bytes(M, max(A if self.continuous else n_out, 32)) // 4 + 64, device=dev)
        idx = torch.empty(E, B, dtype=torch.int32, device=dev)
        for e in range(E):
            worker.wait(e)
            idx[e].copy_(h_idx[e], non_blocking=True)
            for k in range(MB):
                mb = idx[e][k * M:(k + 1) * M]
                x = ctx.gather_rows(obs_flat, mb)
                a_mb = ctx.gather_rows(act_bits, mb)
                lp_mb, adv_mb, ret_mb = ctx.gather_rows(old_logp, mb), ctx.gather_rows(adv_f, mb), ctx.gather_rows(ret_f, mb)
                self.adam_step += 1
                hyper.step = self.adam_step
                self.G.zero_()
                dval = torch.empty(M, device=dev)
                if self.continuous:
                    mean, log_std, val = net.get_means_log_stds_and_values(x)
                    mean_c, ls_c, val_c = mean.contiguous(), log_std.contiguous(), val.contiguous()
                    dmean, dls = torch.empty_like(mean_c), torch.empty_like(ls_c)
                    ctx.ppo_loss_gaussian(mean_c.detach(), ls_c.detach(), val_c.detach(), a_mb, lp_mb, adv_mb, ret_mb, hyper,
                                          losses[e * MB + k], dmean, dls, dval, loss_ws, log_std_row_stride=ls_c.shape[-1])
                    torch.autograd.backward([mean_c, ls_c, val_c], [dmean, dls, dval])
                else:
                    logits, val = net.get_logits_and_values(x)
                    logits_c, val_c = logits.contiguous(), val.contiguous()
                    dlogits = torch.empty_like(logits_c)
                    ctx.ppo_loss_discrete(logits_c.detach(), val_c.detach(), a_mb.view(torch.int32), lp_mb, adv_mb, ret_mb, hyper,
                                          losses[e * MB + k], dlogits, dval, loss_ws)
                    torch.autograd.backward([logits_c, val_c], [dlogits, dval])
                if dist.enabled:
                    dist.all_reduce_sum(self.G)
                    dist.all_reduce_sum(losses[e * MB + k])
                ctx.clip_adam_step(self.P, self.G, self.M, self.V, hyper, self.adam_ws, self.grad_norm)
        worker.finish()
        self._publish_steps()
        self.last_losses = losses


# ------------------------------------------------------------------------------------------------
# Agents
# ------------------------------------------------------------------------------------------------
class _PPOBase(PolicyEvaluation):
    _continuous = False
    _default_network: Any = None

    def _setup(self, env_fn, cfg, network_cls, process_group=None, dp=False, dp_permutation="local", dp_exchange="fused",
               minibatch_permutation="numpy"):
        self.device = _require_cuda()
        self.ctx = N.get_context(self.device.index)
        if cfg.seed is not None:
            np.random.seed(cfg.seed)                                   # ppo.py:120-122
            torch.manual_seed(cfg.seed)
        self._dist = _Dist(process_group, dp, dp_permutation, dp_exchange, minibatch_permutation)
        if self._dist.perm_mode == "numpy":
            self._dist.sync_numpy_stream(self.device)

        self._env_fn = env_fn                                          # evaluate() builds new environments from it
        if getattr(env_fn, "vectorized", False):                       # additive: env_fn(num_envs) -> batched vector env
            self.envs = env_fn(cfg.num_envs)
            # env-sharded data parallelism: this rank simulates global envs [rank*N, (rank+1)*N) -- distinct reset / dynamics
            # draws per shard unless the factory already placed the shard itself
            if self._dist.enabled and getattr(self.envs, "device_resident", False) and self.envs.desc.env_offset == 0:
                self.envs.desc.env_offset = self._dist.rank * cfg.num_envs
        else:
            self.envs = gym.vector.SyncVectorEnv([env_fn for _ in range(cfg.num_envs)], copy=True, autoreset_mode="Disabled")
        obs_space, act_space = self.envs.single_observation_space, self.envs.single_action_space
        self.network = network_cls(obs_space, act_space, cfg=cfg).to(self.device)
        network_parameter_init_(self.network, gain=sqrt(2.0), small_actor_out=not self._continuous)
        if self._dist.enabled:                                          # replicas start from rank 0's parameters
            for p in self.network.parameters():
                self._dist.dist.broadcast(p.data, src=0, group=self._dist.group)

        self.obs_dim = int(np.prod(obs_space.shape))
        self.act_dim = int(np.prod(act_space.shape)) if self._continuous else int(act_space.n)
        if type(self.network) is self._default_network:
            self.engine = FusedMlpEngine(self.ctx, self.network, cfg, self.obs_dim, self.act_dim, self._continuous,
                                         self.device, self._dist)
            self.network.engine = self.engine
        else:
            self.engine = AutogradEngine(self.ctx, self.network, cfg, self._continuous, self.device, self._dist)

        self.optimizer = torch.optim.Adam(self.network.parameters(), lr=cfg.lr, eps=cfg.adam_eps)       # ppo.py:135
        self.engine.bind_optimizer(self.optimizer)
        self.lr_scheduler = torch.optim.lr_scheduler.LinearLR(                                          # ppo.py:137-142
            self.optimizer, start_factor=1.0, end_factor=0.05 if cfg.decay_lr else 1.0,
            total_iters=cfg.total_steps // (cfg.num_envs * cfg.rollout_steps))
        self.logger = Logger()
        self.timer = Timer()
        self.checkpointer = Checkpointer(folder="models", run_name="default")
        self.ticker = Ticker(cfg.total_steps, cfg.num_envs, cfg.rollout_steps, verbose=cfg.verbose)
        self.cfg = cfg
        self._buffer = None
        self._rollout_graph, self._rollout_seen = None, None
        self._epstats = None

    # ---- rollout (ppo.py:153-186) -------------------------------------------------------------------
    def rollout(self) -> RolloutBuffer:
        """Collect one rollout; returns the device-resident buffer (list-like for user code)."""
        cfg = self.cfg
        if self._buffer is None:
            self._buffer = RolloutBuffer(self.ctx, cfg.rollout_steps, cfg.num_envs, self.obs_dim,
                                         self.act_dim if self._continuous else 1, self._continuous, self.device)
        buf = self._buffer
        buf.filled = 0
        if getattr(self.envs, "device_resident", False) and isinstance(self.engine, FusedMlpEngine):
            # device-resident environments: sampling kernel -> environment kernel per step, nothing crosses PCIe
            envs = self.envs
            if getattr(buf, "values", None) is None:
                buf.values = torch.empty(buf.T, buf.N, dtype=torch.float32, device=self.device)
                buf.logp = torch.empty(buf.T, buf.N, dtype=torch.float32, device=self.device)
                if getattr(envs, "normalize_reward", False):            # rewards are normalised: keep the raw ones for the Ticker
                    buf.raw_rewards = torch.empty(buf.T, buf.N, dtype=torch.float32, device=self.device)
            buf.policy_stamp = None
            stamp = self.engine.policy_stamp()
            # From the third rollout into the same buffers the T x (forward, head, sampling, environment) launches are replayed
            # as ONE CUDA graph; the draw counters baked into it are relative, their base lives on the device.
            gkey = (buf.obs.data_ptr(), buf.values.data_ptr(), envs.cur_obs.data_ptr(), self.engine.P.data_ptr(), cfg.rollout_steps)
            rg = self._rollout_graph
            if rg is not None and rg["key"] == gkey:
                rg["base"].fill_(self.engine.draws)
                rg["graph"].replay()
                self.engine.draws += cfg.rollout_steps
                self.ctx.count_launches(rg["launches"])
            elif self.engine.use_graphs and self._rollout_seen == gkey:
                base = torch.zeros(1, dtype=torch.int64, device=self.device)
                graph = torch.cuda.CUDAGraph()
                torch.cuda.synchronize()
                l0 = self.ctx.launches
                self.ctx.set_draw_counter_base(base)
                try:
                    with torch.cuda.graph(graph):
                        for step_idx in range(cfg.rollout_steps):
                            envs.step_into(buf, step_idx, self.engine.sample_actions_device(envs.cur_obs, buf.values[step_idx],
                                                                                            buf.logp[step_idx], counter=step_idx))
                finally:
                    self.ctx.set_draw_counter_base(None)
                self._rollout_graph = rg = dict(key=gkey, graph=graph, base=base, launches=self.ctx.launches - l0)
                base.fill_(self.engine.draws)
                graph.replay()
                self.engine.draws += cfg.rollout_steps
            else:
                self._rollout_seen = gkey
                for step_idx in range(cfg.rollout_steps):
                    envs.step_into(buf, step_idx, self.engine.sample_actions_device(envs.cur_obs, buf.values[step_idx], buf.logp[step_idx]))
            if self.engine.policy_stamp() == stamp:
                buf.policy_stamp = stamp                               # V(obs), log_prob(action) of exactly these parameters
            if self.ticker is not None:                                # episode statistics on the device, read lazily (no sync here)
                self._device_episode_stats(buf)
            self.current_observations = envs.cur_obs
            return buf
        observations = self.current_observations
        for step_idx in range(cfg.rollout_steps):
            actions = self.network.get_actions(observations, device=self.device)
            next_observations, rewards, terminations, truncations, infos = self.envs.step(actions)
            tick_rewards = infos.get("raw_rewards", rewards) if isinstance(infos, dict) else rewards   # raw, if the env normalises
            buf.store(step_idx, observations, next_observations, actions, rewards, terminations, truncations)
            dones = np.logical_or(terminations, truncations)
            if np.any(dones):                                          # autoreset disabled: masked reset (ppo.py:174-179)
                observations, infos = self.envs.reset(options={"reset_mask": dones})
            else:
                observations = next_observations
            if self.ticker is not None:
                self.ticker.tick(tick_rewards, dones)
        self.current_observations = observations
        return buf

    # ---- evaluation (diamond/evaluation.py) --------------------------------------------------------------------------
    def predict(self, observations, deterministic: bool = True):
        """Actions of the current policy for observations [n, obs_dim]: a host array in, a NumPy array out; a device tensor in, a
        device tensor out.  deterministic=True: the greedy action (the first argmax of the logits, or the Gaussian means, not
        clipped); False: a draw of the evaluation generator (its own key and counter: the training sampling counter and the numpy /
        torch streams do not move).  Default networks run the fused forward and the greedy / sampling kernels; a custom
        network_cls runs its get_logits_and_values / get_means_log_stds_and_values under inference_mode."""
        obs = as_device_obs(observations, self.obs_dim, self.device)
        n = obs.shape[0]
        eng, log_std = self.engine, None
        if getattr(eng, "fused", False):
            head = torch.empty(n, eng.A, dtype=torch.float32, device=self.device)
            self.ctx.mlp_forward(eng.fm.desc, eng.P, obs, n, 1, head, None, eng.fwd_ws)
            if self._continuous:
                log_std = eng.P[eng.fm.layout.log_std:eng.fm.layout.log_std + eng.A]
        else:
            with torch.inference_mode():
                if self._continuous:
                    head, log_stds, _ = self.network.get_means_log_stds_and_values(obs)
                    log_std = shared_log_std(log_stds)
                else:
                    head, _ = self.network.get_logits_and_values(obs)
                head = head.reshape(n, -1).contiguous()
        key, counter = self._eval_draw() if not deterministic else (0, 0)
        actions = select_actions(self.ctx, head, log_std, deterministic, key, counter, greedy_kernel=getattr(eng, "fused", False))
        return actions if torch.is_tensor(observations) else actions.cpu().numpy()

    # ---- episode statistics of device-resident rollouts (utils.py:99-123 without the per-step host loop) ------------
    def _device_episode_stats(self, buf):
        """Ticker bookkeeping of this rollout in two kernels (dppo_episode_stats); the ~100 numbers the Ticker needs are copied to
        pinned memory asynchronously and consumed at the next rollout / when `ticker.logs` is read -- the host never waits for
        the rollout between rollout() and learn()."""
        st = self._epstats
        W, dev = self.ticker.window_size, self.device
        if st is None or st["N"] != buf.N or st["T"] != buf.T or st["W"] != W:
            st = self._epstats = dict(N=buf.N, T=buf.T, W=W, pending=None,
                                      ep_return=torch.zeros(buf.N, dtype=torch.float64, device=dev),
                                      ep_len=torch.zeros(buf.N, dtype=torch.int32, device=dev),
                                      out=torch.zeros(W + 2, dtype=torch.float64, device=dev),        # [returns W | finished | kept]
                                      out_len=torch.zeros(W, dtype=torch.int32, device=dev), out_n=torch.zeros(1, dtype=torch.int32, device=dev),
                                      finished=torch.zeros(1, dtype=torch.int64, device=dev),
                                      ws=torch.empty(self.ctx.episode_stats_workspace_bytes(buf.T, buf.N) + 8, dtype=torch.uint8, device=dev),
                                      h_out=torch.zeros(W + 2, dtype=torch.float64).pin_memory(), h_len=torch.zeros(W, dtype=torch.int32).pin_memory())
            self.ticker._flush_pending = self._flush_episode_stats
            pend = getattr(self, "_pending_epstats", None)             # resumed run: running returns / lengths of open episodes
            if pend is not None and pend["ep_len"].numel() == buf.N:
                st["ep_return"].copy_(pend["ep_return"]); st["ep_len"].copy_(pend["ep_len"])
            self._pending_epstats = None
        self._flush_episode_stats()                                    # the previous rollout's numbers (long since copied)
        rewards = getattr(buf, "raw_rewards", None)                    # a reward-normalising environment's raw rewards
        self.ctx.episode_stats(buf.rewards if rewards is None else rewards, buf.terminations, buf.truncations, st["ep_return"], st["ep_len"], W, st["out"][:W],
                               st["out_len"], st["out_n"], st["finished"], st["ws"])
        st["out"][W:W + 1].copy_(st["finished"])
        st["out"][W + 1:W + 2].copy_(st["out_n"])
        st["h_out"].copy_(st["out"], non_blocking=True)
        st["h_len"].copy_(st["out_len"], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        st["pending"] = dict(event=ev, steps=buf.T)

    def _flush_episode_stats(self):
        st = self._epstats
        if st is None or st["pending"] is None:
            return
        pend, st["pending"] = st["pending"], None
        pend["event"].synchronize()
        W = st["W"]
        finished, kept = int(st["h_out"][W]), int(st["h_out"][W + 1])
        self.ticker.tick_rollout(pend["steps"], finished, st["h_out"][:kept].tolist(), st["h_len"][:kept].tolist())

    # ---- GAE (ppo.py:188-222) -----------------------------------------------------------------------
    def calculate_advantage(self, rewards, terminations, truncations, values, next_values) -> torch.Tensor:
        """Generalised Advantage Estimation on the GPU (dppo_gae_f32); [T, N] float32 tensors in, [T, N] out."""
        args = [torch.as_tensor(x).to(self.device, torch.float32).contiguous() for x in
                (rewards, terminations, truncations, values, next_values)]
        return self.ctx.gae(*args, self.cfg.gamma, self.cfg.gae_lambda)

    # ---- learn (ppo.py:224-287) ----------------------------------------------------------------------
    def learn(self, experience, events=None) -> None:
        """Update policy and value networks from a rollout: either the RolloutBuffer `rollout()`
        returned, or a reference-style list of per-step NumPy arrays."""
        buf = experience if isinstance(experience, RolloutBuffer) else \
            RolloutBuffer.from_lists(self.ctx, experience, self._continuous, self.device)
        self.engine.learn(buf, events)
        self.optimizer._opt_called = True                              # the kernels performed the optimiser steps
        self.lr_scheduler.step()                                       # ppo.py:287

    @property
    def last_losses(self):
        """[E*MB, 4] device tensor: policy, value, entropy, total loss of every minibatch of the last learn()."""
        return self.engine.last_losses

    # ---- train (ppo.py:289-312) ----------------------------------------------------------------------
    # ---- train-level checkpoint state (SURVEY.md 8 f3: the resume path the reference lacks) ---------------------------
    def _train_state(self, rollouts_done: int) -> dict:
        """Everything beyond {"model_state", "opt_state"} that a bit-identical continuation of train() needs: position in the
        run, LR schedule, the numpy global stream (minibatch permutations) and torch CPU stream, the engine's counter-based
        generators, the environments and the Ticker."""
        eng, envs = self.engine, self.envs
        st = dict(version=1, rollouts_done=int(rollouts_done), lr_scheduler=self.lr_scheduler.state_dict(),
                  numpy_state=np.random.get_state(legacy=True), torch_rng=torch.get_rng_state(),
                  engine={k: getattr(eng, k) for k in ("draws", "seed", "perm_counter", "perm_seed") if hasattr(eng, k)})
        self._flush_episode_stats()
        tk = self.ticker
        if tk is not None:
            st["ticker"] = dict(current_step=tk.current_step, current_episode=tk.current_episode, returns=list(tk.recent_returns),
                                lengths=list(tk.recent_lengths), current_returns=tk.current_returns.copy(),
                                current_lengths=tk.current_lengths.copy(), elapsed=time.time() - tk.start_time)
        if self._epstats is not None:
            st["epstats"] = dict(ep_return=self._epstats["ep_return"].cpu(), ep_len=self._epstats["ep_len"].cpu())
        if getattr(envs, "device_resident", False):
            st["envs"] = dict(kind="device", seed=int(envs.desc.seed), env_offset=int(envs.desc.env_offset),
                              update_running_mean=envs.update_running_mean,           # + normalisation statistics, if any
                              **{k: getattr(envs, k).cpu() for k in envs.state_tensors})
        else:
            import pickle
            try:                                                       # host environments: whatever pickles (the in-repo shim does)
                st["envs"] = dict(kind="pickle", blob=pickle.dumps(envs), obs=np.asarray(self.current_observations).copy())
            except Exception:
                st["envs"] = dict(kind="none")
        return st

    def _restore_train_state(self, st: dict) -> int:
        if st.get("version") != 1:
            raise ValueError("unknown train_state version in checkpoint")
        self.lr_scheduler.load_state_dict(st["lr_scheduler"])
        lr = self.lr_scheduler.get_last_lr()[0]
        for g in self.optimizer.param_groups:
            g["lr"] = lr
        np.random.set_state(st["numpy_state"])
        torch.set_rng_state(st["torch_rng"])
        for k, v in st["engine"].items():
            setattr(self.engine, k, v)
        tk, ts = self.ticker, st.get("ticker")
        if tk is not None and ts is not None:
            tk.current_step, tk.current_episode = ts["current_step"], ts["current_episode"]
            tk.recent_returns.clear(); tk.recent_returns.extend(ts["returns"])
            tk.recent_lengths.clear(); tk.recent_lengths.extend(ts["lengths"])
            tk.current_returns[:] = ts["current_returns"]; tk.current_lengths[:] = ts["current_lengths"]
            tk.start_time = time.time() - ts["elapsed"]
        self._pending_epstats = st.get("epstats")                      # adopted when the device accumulators are created
        es = st["envs"]
        if es["kind"] == "device":
            envs = self.envs
            envs.desc.seed, envs.desc.env_offset = es["seed"], es["env_offset"]
            for k in envs.state_tensors:
                getattr(envs, k).copy_(es[k])
            if "update_running_mean" in es:
                envs.update_running_mean = es["update_running_mean"]
            self.current_observations = envs.cur_obs
        elif es["kind"] == "pickle":
            import pickle
            self.envs = pickle.loads(es["blob"])
            self.current_observations = es["obs"]
        else:
            raise RuntimeError("the checkpoint holds no environment state (the environments could not be pickled): cannot resume")
        return int(st["rollouts_done"])

    def save_checkpoint(self, rollouts_done: int):
        """Reference payload keys (utils.py:584-600: step, model_state, opt_state) + "train_state" for resume."""
        env_steps = rollouts_done * self.cfg.rollout_steps * self.cfg.num_envs
        return self.checkpointer.save(env_steps, self.network, self.optimizer, extra={"train_state": self._train_state(rollouts_done)})

    # ---- train (ppo.py:289-312) ----------------------------------------------------------------------
    def train(self, *, resume_from=None, max_rollouts: int | None = None) -> None:
        """The reference's training loop.  Additive: `resume_from=<checkpoint path>` continues an interrupted run (model, Adam
        moments and step, LR schedule, RNG streams, environments, Ticker) so that it ends bit-identical to an uninterrupted
        one; `max_rollouts` stops after that many rollouts of THIS call, saving a checkpoint (interruption point for tests)."""
        cfg = self.cfg
        first = 0
        if resume_from is not None:
            chk = torch.load(resume_from, map_location="cpu", weights_only=False)
            if "train_state" not in chk:
                raise ValueError(f"{resume_from} has no train_state: it was not written by train() of this package")
            self.network.load_state_dict(chk["model_state"])
            self.optimizer.load_state_dict(chk["opt_state"])
            if hasattr(self.engine, "_resync_optimizer"):
                self.engine._resync_optimizer()
            first = self._restore_train_state(chk["train_state"])
        else:
            # under data parallelism the shards are different environments of one global run: host vector envs seed sub-env i
            # with seed + i (Gymnasium), so rank r starts at seed + r*N; device envs key their draws by global env id (env_offset)
            seed = cfg.seed
            if seed is not None and self._dist.enabled and not getattr(self.envs, "device_resident", False):
                seed = cfg.seed + self._dist.rank * cfg.num_envs
            self.current_observations, _ = self.envs.reset(seed=seed)
            if self._epstats is not None:                              # fresh environments: running returns / lengths restart
                self._flush_episode_stats()
                self._epstats["ep_return"].zero_()
                self._epstats["ep_len"].zero_()
        last_checkpoint_time = time.time()
        total_rollouts = cfg.total_steps // (cfg.rollout_steps * cfg.num_envs)
        stop = total_rollouts if max_rollouts is None else min(total_rollouts, first + max_rollouts)
        done = first
        for rollout_idx in range(first, stop):
            experience = self.rollout()
            self.learn(experience)
            done = rollout_idx + 1
            if cfg.checkpoint and self._dist.rank == 0 and time.time() - last_checkpoint_time >= cfg.save_interval:
                self.save_checkpoint(done)                             # replicas are identical: rank 0 writes
                last_checkpoint_time = time.time()
        if (cfg.checkpoint or max_rollouts is not None) and done > first and self._dist.rank == 0:
            self.last_checkpoint = self.save_checkpoint(done)
        self._flush_episode_stats()
        if hasattr(self.engine, "check_health"):
            torch.cuda.current_stream().synchronize()
            self.engine.check_health()
        if stop == total_rollouts:
            self.envs.close()


class PPO(_PPOBase):
    """Discrete-action PPO (reference: diamond/ppo.py:111-312)."""
    _continuous = False
    _default_network = ActorCriticNetwork

    def __init__(self, env_fn: Callable[[], Any], cfg: PPOConfig = PPOConfig(), network_cls: Any = ActorCriticNetwork,
                 *, process_group=None, dp: bool = False, dp_permutation: str = "local", dp_exchange: str = "fused",
                 minibatch_permutation: str = "numpy") -> None:
        self._setup(env_fn, cfg, network_cls, process_group, dp, dp_permutation, dp_exchange, minibatch_permutation)
        self.current_step = 0


class ContinuousPPO(_PPOBase):
    """Gaussian-policy PPO (reference: diamond/continuous_ppo.py:124-324)."""
    _continuous = True
    _default_network = ContinuousActorCriticNetwork

    def __init__(self, env_fn: Callable[[], Any], cfg: ContinuousPPOConfig = ContinuousPPOConfig(),
                 network_cls: Any = ContinuousActorCriticNetwork, *, process_group=None, dp: bool = False,
                 dp_permutation: str = "local", dp_exchange: str = "fused", minibatch_permutation: str = "numpy") -> None:
        self._setup(env_fn, cfg, network_cls, process_group, dp, dp_permutation, dp_exchange, minibatch_permutation)
