"""ctypes binding of libdppo.so (include/dppo.h) — the only way the package reaches the GPU.

There is no fallback: if the library has not been built, or no sm_100 device is present when a
context is requested, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdppo.so")


class NativeError(RuntimeError):
    pass


class MlpDesc(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("hidden", C.c_int32), ("act_dim", C.c_int32), ("continuous", C.c_int32)]


class MlpLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("w1", "b1", "w2", "b2", "w3", "b3", "wa", "ba", "wc", "bc", "log_std", "total")]


class RnnDesc(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("hidden", C.c_int32), ("gru_hidden", C.c_int32), ("act_dim", C.c_int32), ("continuous", C.c_int32)]


class RnnLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("w1", "b1", "wih", "whh", "bih", "bhh", "w3", "b3", "wa", "ba", "wc", "bc", "log_std", "total")]


class EnvDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("num_envs", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("seed", C.c_uint64),
                ("env_offset", C.c_int64), ("p_term", C.c_float), ("p_trunc", C.c_float),
                ("normalize", C.c_int32), ("pad0", C.c_int32), ("gamma", C.c_double), ("epsilon", C.c_double),
                ("clip_observation", C.c_double), ("clip_reward", C.c_double)]


ENV_NORMALIZE_OBS, ENV_NORMALIZE_REWARD = 1, 2     # dppo_env_desc.normalize bits


class EnvState(C.Structure):
    _fields_ = [("state", C.c_void_p), ("steps", C.c_void_p), ("episode", C.c_void_p), ("ep_return", C.c_void_p), ("cur_obs", C.c_void_p),
                ("obs_mean", C.c_void_p), ("obs_var", C.c_void_p), ("obs_count", C.c_void_p), ("ret_stats", C.c_void_p),
                ("update", C.c_void_p)]


class Hyper(C.Structure):
    _fields_ = [("ppo_clip", C.c_float), ("value_loss_weight", C.c_float), ("entropy_beta", C.c_float),
                ("grad_norm_clip", C.c_float), ("adam_eps", C.c_float), ("pad0", C.c_float),
                ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("step", C.c_int64),
                ("advantage_norm", C.c_int32), ("pad1", C.c_int32), ("adv_count", C.c_int64),
                ("loss_denominator", C.c_int64), ("step_consts", C.c_void_p), ("grad_sumsq", C.c_void_p)]


# every symbol include/dppo.h declares (tests/test_abi.py checks the header against this list)
EXPORTS = [
    "dppo_create", "dppo_destroy", "dppo_last_error", "dppo_version", "dppo_device_info", "dppo_set_option", "dppo_launch_count", "dppo_count_launches",
    "dppo_buffer_store_step", "dppo_step_record_bytes", "dppo_sample_categorical", "dppo_sample_gaussian",
    "dppo_gae_f32", "dppo_adv_normalize_f32", "dppo_permutation_mt19937", "dppo_permutation_mt19937_skip", "dppo_mt19937_seed",
    "dppo_gather_rows_f32", "dppo_mlp_layout_compute", "dppo_mlp_workspace_bytes", "dppo_mlp_forward", "dppo_mlp_next_values", "dppo_mlp_next_values_workspace_bytes",
    "dppo_logprob_categorical", "dppo_logprob_gaussian", "dppo_mlp_grad_minibatch", "dppo_mlp_fused_heads_supported",
    "dppo_mlp_gemm_heads_workspace_bytes", "dppo_mlp_grad_minibatch_gemm_heads", "dppo_small_update", "dppo_small_update_supported", "dppo_clip_adam_step",
    "dppo_clip_adam_workspace_bytes", "dppo_grad_sumsq_bytes", "dppo_ppo_loss_discrete", "dppo_ppo_loss_gaussian",
    "dppo_ppo_loss_workspace_bytes", "dppo_fma_peak_kernel", "dppo_tc_linear_f32", "dppo_tc_linear_workspace_bytes",
    "dppo_tc_colsum_parts", "dppo_tc_wgrad_f32", "dppo_tc_wgrad_workspace_bytes", "dppo_tc_mma_probe", "dppo_dp_create", "dppo_dp_handle_bytes", "dppo_dp_handle", "dppo_dp_connect", "dppo_dp_destroy", "dppo_dp_status",
    "dppo_permutation_device", "dppo_perm_shard_filter", "dppo_dp_slot", "dppo_dp_zero_slot", "dppo_dp_workspace_bytes", "dppo_dp_allreduce_clip_adam",
    "dppo_env_reset", "dppo_env_step", "dppo_set_draw_counter_base", "dppo_episode_stats", "dppo_episode_stats_workspace_bytes",
    "dppo_select_greedy_categorical", "dppo_eval_episodes",
    "dppo_rnn_layout_compute", "dppo_rnn_workspace_bytes", "dppo_rnn_forward", "dppo_rnn_grad_minibatch",
]

_lib = None
_lib_lock = threading.Lock()


def load_library() -> C.CDLL:
    """Loads libdppo.so (built in-tree by `make -C diamond-ppo_b200` / __graft_entry__.build())."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeError(f"{LIB_PATH} not found: build it with `make -C {os.path.dirname(_HERE)}` "
                                  "(python __graft_entry__.py build). There is no fallback path.")
            lib = C.CDLL(LIB_PATH)
            lib.dppo_last_error.restype = C.c_char_p
            lib.dppo_last_error.argtypes = [C.c_void_p]
            for name in ("dppo_step_record_bytes", "dppo_mlp_workspace_bytes", "dppo_clip_adam_workspace_bytes", "dppo_grad_sumsq_bytes",
                         "dppo_ppo_loss_workspace_bytes", "dppo_tc_linear_workspace_bytes", "dppo_tc_wgrad_workspace_bytes", "dppo_launch_count", "dppo_dp_workspace_bytes", "dppo_grad_sumsq_bytes",
                         "dppo_rnn_workspace_bytes", "dppo_episode_stats_workspace_bytes", "dppo_mlp_next_values_workspace_bytes",
                         "dppo_mlp_gemm_heads_workspace_bytes"):
                getattr(lib, name).restype = C.c_int64
            lib.dppo_dp_slot.restype = C.c_void_p
            _lib = lib
    return _lib


def _ptr(t):
    if t is None:
        return C.c_void_p(0)
    if isinstance(t, int):                      # raw device pointer (e.g. a slot of the DP exchange buffer)
        return C.c_void_p(t)
    if isinstance(t, torch.Tensor):
        assert t.is_contiguous(), "libdppo takes contiguous tensors"
        return C.c_void_p(t.data_ptr())
    if isinstance(t, np.ndarray):
        assert t.flags["C_CONTIGUOUS"]
        return C.c_void_p(t.ctypes.data)
    raise TypeError(type(t))


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def mlp_layout(desc: MlpDesc) -> MlpLayout:
    lay = MlpLayout()
    if load_library().dppo_mlp_layout_compute(C.byref(desc), C.byref(lay)):
        raise NativeError("dppo_mlp_layout_compute: bad descriptor")
    return lay


def rnn_layout(desc: RnnDesc) -> RnnLayout:
    lay = RnnLayout()
    if load_library().dppo_rnn_layout_compute(C.byref(desc), C.byref(lay)):
        raise NativeError("dppo_rnn_layout_compute: bad descriptor")
    return lay


# ---- host-only entry points (usable without a GPU) -------------------------------------------
def fused_heads_supported(desc: MlpDesc) -> bool:
    """dppo_mlp_fused_heads_supported: whether dppo_mlp_grad_minibatch's fused head kernel takes this network shape."""
    return bool(load_library().dppo_mlp_fused_heads_supported(C.byref(desc)))


def mt19937_seed(seed: int):
    key = np.zeros(624, np.uint32)
    pos = C.c_int32(0)
    load_library().dppo_mt19937_seed(_ptr(key), C.byref(pos), C.c_uint32(seed & 0xFFFFFFFF))
    return key, pos.value


def permutation_mt19937(key: np.ndarray, pos: int, n: int, out: np.ndarray | None = None):
    """np.random.permutation(n) continued from MT19937 state (key, pos); returns (int32 perm, new pos)."""
    assert key.dtype == np.uint32 and key.size == 624 and key.flags["C_CONTIGUOUS"]
    if out is None:
        out = np.empty(n, np.int32)
    assert out.dtype == np.int32 and out.size >= n
    p = C.c_int32(pos)
    rc = load_library().dppo_permutation_mt19937(_ptr(key), C.byref(p), C.c_int64(n), _ptr(out))
    if rc:
        raise NativeError("dppo_permutation_mt19937: bad arguments")
    return out, p.value


def permutation_mt19937_skip(key: np.ndarray, pos: int, n: int) -> int:
    """Advances (key, pos) exactly as permutation_mt19937(key, pos, n) would, without building the permutation; returns the new pos."""
    assert key.dtype == np.uint32 and key.size == 624 and key.flags["C_CONTIGUOUS"]
    p = C.c_int32(pos)
    if load_library().dppo_permutation_mt19937_skip(_ptr(key), C.byref(p), C.c_int64(n)):
        raise NativeError("dppo_permutation_mt19937_skip: bad arguments")
    return p.value


def numpy_global_permutations(n: int, count: int, outs=None):
    """`count` consecutive np.random.permutation(n) draws from numpy's global legacy RandomState
    (diamond/ppo.py:254), generated by libdppo and with the global stream advanced exactly as numpy
    would have advanced it."""
    st = np.random.get_state(legacy=True)
    assert st[0] == "MT19937"
    key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
    pos = int(st[2])
    res = []
    for i in range(count):
        out, pos = permutation_mt19937(key, pos, n, None if outs is None else outs[i])
        res.append(out)
    np.random.set_state(("MT19937", key, pos, st[3], st[4]))
    return res


class Context:
    """Owns a dppo_ctx for one CUDA device."""

    def __init__(self, device: int | None = None):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise NativeError("libdppo needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.cuda.current_device() if device is None else int(device)
        h = C.c_void_p()
        rc = self.lib.dppo_create(C.byref(h), C.c_int(self.device))
        if rc:
            raise NativeError(self.lib.dppo_last_error(None).decode())
        self.h = h
        sm, maj, mnr = C.c_int(), C.c_int(), C.c_int()
        self.lib.dppo_device_info(self.h, C.byref(sm), C.byref(maj), C.byref(mnr))
        self.sm_count, self.cc = sm.value, (maj.value, mnr.value)
        self._launch_base = 0

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.dppo_destroy(self.h)
                self.h = None
        except Exception:
            pass

    @property
    def launches(self) -> int:
        """Kernels launched through this context (counted inside libdppo at every launch; bench.py's gpu_launches)."""
        return int(self.lib.dppo_launch_count(self.h))

    @launches.setter
    def launches(self, _):          # the old Python-side estimates (`self.launches += n`) are ignored
        pass

    def count_launches(self, n: int):
        """Adds launches that were replayed from a CUDA graph captured through this context."""
        self.lib.dppo_count_launches(self.h, C.c_int64(int(n)))

    def set_option(self, name: str, value: int):
        self._check(self.lib.dppo_set_option(self.h, name.encode(), C.c_int(int(value))), "dppo_set_option")

    def _check(self, rc, what):
        if rc:
            raise NativeError(f"{what}: {self.lib.dppo_last_error(self.h).decode()}")

    # ---- GAE -------------------------------------------------------------------------------
    def gae(self, rewards, terminations, truncations, values, next_values, gamma, gae_lambda, advantages=None, inputs_settled=False,
            returns=None, stats=None):
        T, N = rewards.shape
        if advantages is None:
            advantages = torch.empty_like(rewards)
        # inputs_settled (include/dppo.h): False -- plain launch, nothing requested early (any caller); "rollout" -- the kernel
        # launched just before this call writes none of rewards / terminations / truncations; True -- none of the five inputs
        level = 1 if inputs_settled == "rollout" else (2 if inputs_settled else 0)
        self.lib.dppo_set_option(self.h, b"gae_inputs_settled", C.c_int(level))
        self._check(self.lib.dppo_gae_f32(self.h, _ptr(rewards), _ptr(terminations), _ptr(truncations), _ptr(values),
                                          _ptr(next_values), _ptr(advantages), _ptr(returns), _ptr(stats), C.c_int(T),
                                          C.c_int(N), C.c_double(gamma), C.c_double(gae_lambda), _stream()), "dppo_gae_f32")
        self.launches += 1
        return advantages

    def adv_normalize(self, adv, stats, count, out=None):
        out = torch.empty_like(adv) if out is None else out
        self._check(self.lib.dppo_adv_normalize_f32(self.h, _ptr(adv), _ptr(out), _ptr(stats), C.c_int64(count),
                                                    C.c_int64(adv.numel()), _stream()), "dppo_adv_normalize_f32")
        self.launches += 1
        return out

    # ---- rollout ---------------------------------------------------------------------------
    def step_record_bytes(self, N, D, A, continuous):
        return int(self.lib.dppo_step_record_bytes(C.c_int(N), C.c_int(D), C.c_int(A), C.c_int(int(continuous))))

    def buffer_store_step(self, record, t, N, D, A, continuous, obs, next_obs, actions, rewards, terms, truncs):
        self._check(self.lib.dppo_buffer_store_step(self.h, _ptr(record), C.c_int(t), C.c_int(N), C.c_int(D), C.c_int(A),
                                                    C.c_int(int(continuous)), _ptr(obs), _ptr(next_obs), _ptr(actions),
                                                    _ptr(rewards), _ptr(terms), _ptr(truncs), _stream()), "dppo_buffer_store_step")
        self.launches += 1

    def sample_categorical(self, logits, seed, counter, env_offset=0, actions=None, log_probs=None):
        N, A = logits.shape
        actions = torch.empty(N, dtype=torch.int64, device=logits.device) if actions is None else actions
        self._check(self.lib.dppo_sample_categorical(self.h, _ptr(logits), C.c_int(N), C.c_int(A), C.c_uint64(seed),
                                                     C.c_uint64(counter), C.c_int64(env_offset), _ptr(actions),
                                                     _ptr(log_probs), _stream()), "dppo_sample_categorical")
        self.launches += 1
        return actions

    def sample_gaussian(self, mean, log_std, seed, counter, env_offset=0, actions=None, log_probs=None):
        N, A = mean.shape
        actions = torch.empty_like(mean) if actions is None else actions
        self._check(self.lib.dppo_sample_gaussian(self.h, _ptr(mean), _ptr(log_std), C.c_int(N), C.c_int(A),
                                                  C.c_uint64(seed), C.c_uint64(counter), C.c_int64(env_offset),
                                                  _ptr(actions), _ptr(log_probs), _stream()), "dppo_sample_gaussian")
        self.launches += 1
        return actions

    def select_greedy_categorical(self, logits, actions=None, log_probs=None):
        """torch.argmax(logits, -1) (first maximum, NaN counts as the maximum) -> int64 [N] (dppo_select_greedy_categorical)."""
        N, A = logits.shape
        actions = torch.empty(N, dtype=torch.int64, device=logits.device) if actions is None else actions
        self._check(self.lib.dppo_select_greedy_categorical(self.h, _ptr(logits), C.c_int(N), C.c_int(A), _ptr(actions), _ptr(log_probs),
                                                            _stream()), "dppo_select_greedy_categorical")
        return actions

    def set_draw_counter_base(self, counter_base):
        """counter_base: device int64/uint64 tensor [1] (None clears); added to every sampling draw counter at run time."""
        self._check(self.lib.dppo_set_draw_counter_base(self.h, _ptr(counter_base)), "dppo_set_draw_counter_base")

    # ---- MLP -------------------------------------------------------------------------------
    def mlp_workspace_bytes(self, desc, rows, training):
        return int(self.lib.dppo_mlp_workspace_bytes(C.byref(desc), C.c_int64(rows), C.c_int(int(training))))

    def mlp_forward(self, desc, params, obs, rows, heads, head_out, values, ws, idx=None):
        self._check(self.lib.dppo_mlp_forward(self.h, C.byref(desc), _ptr(params), _ptr(obs), _ptr(idx), C.c_int64(rows),
                                              C.c_int(heads), _ptr(head_out), _ptr(values), _ptr(ws),
                                              C.c_int64(ws.numel() * ws.element_size()), _stream()), "dppo_mlp_forward")
        per_row = 16 * desc.hidden
        chunk = max(1, min(rows, (ws.numel() * ws.element_size() - 768) // per_row))
        self.launches += 4 * ((rows + chunk - 1) // chunk)

    def logprob_categorical(self, logits, actions_i32, out):
        rows, A = logits.shape
        self._check(self.lib.dppo_logprob_categorical(self.h, _ptr(logits), _ptr(actions_i32), _ptr(out), C.c_int64(rows),
                                                      C.c_int(A), _stream()), "dppo_logprob_categorical")
        self.launches += 1

    def mlp_next_values_workspace_bytes(self, desc, T, N):
        return int(self.lib.dppo_mlp_next_values_workspace_bytes(C.byref(desc), C.c_int(T), C.c_int(N)))

    def mlp_next_values(self, desc, params, next_obs, terminations, truncations, values, next_values, ws):
        """next_values from recorded rollout values + the critic on final observations only; row selection on the device, no sync."""
        T, N = values.shape
        self._check(self.lib.dppo_mlp_next_values(self.h, C.byref(desc), _ptr(params), _ptr(next_obs), _ptr(terminations), _ptr(truncations),
                                                  _ptr(values), C.c_int(T), C.c_int(N), _ptr(next_values), _ptr(ws),
                                                  C.c_int64(ws.numel() * ws.element_size()), _stream()), "dppo_mlp_next_values")
        self.launches += 8

    def logprob_gaussian(self, mean, log_std, actions, out):
        rows, A = mean.shape
        self._check(self.lib.dppo_logprob_gaussian(self.h, _ptr(mean), _ptr(log_std), _ptr(actions), _ptr(out),
                                                   C.c_int64(rows), C.c_int(A), _stream()), "dppo_logprob_gaussian")
        self.launches += 1

    def mlp_grad_minibatch(self, desc, params, grads, obs, actions, old_logp, adv, returns, adv_stats, idx, M, hyper,
                           losses, ws):
        self._check(self.lib.dppo_mlp_grad_minibatch(self.h, C.byref(desc), _ptr(params), _ptr(grads), _ptr(obs),
                                                     _ptr(actions), _ptr(old_logp), _ptr(adv), _ptr(returns),
                                                     _ptr(adv_stats), _ptr(idx), C.c_int64(M), C.byref(hyper),
                                                     _ptr(losses), _ptr(ws), C.c_int64(ws.numel() * ws.element_size()),
                                                     _stream()), "dppo_mlp_grad_minibatch")
        self.launches += 10

    # ---- GEMM heads: every shape up to DPPO_GEMM_HEADS_MAX_HIDDEN / _ACT (include/dppo.h) ---------------------------------
    def mlp_fused_heads_supported(self, desc) -> bool:
        """True exactly for the shapes the fused head kernel of mlp_grad_minibatch accepts."""
        return fused_heads_supported(desc)

    def mlp_gemm_heads_workspace_bytes(self, desc, rows):
        return int(self.lib.dppo_mlp_gemm_heads_workspace_bytes(C.byref(desc), C.c_int64(rows)))

    def mlp_grad_minibatch_gemm_heads(self, desc, params, grads, obs, actions, old_logp, adv, returns, adv_stats, idx, M, hyper,
                                      losses, ws):
        """mlp_grad_minibatch with the heads as GEMMs around the wide loss kernel (same gradient layout and losses)."""
        self._check(self.lib.dppo_mlp_grad_minibatch_gemm_heads(self.h, C.byref(desc), _ptr(params), _ptr(grads), _ptr(obs),
                                                                _ptr(actions), _ptr(old_logp), _ptr(adv), _ptr(returns),
                                                                _ptr(adv_stats), _ptr(idx), C.c_int64(M), C.byref(hyper),
                                                                _ptr(losses), _ptr(ws), C.c_int64(ws.numel() * ws.element_size()),
                                                                _stream()), "dppo_mlp_grad_minibatch_gemm_heads")
        self.launches += 13

    def small_update_supported(self, desc) -> bool:
        return bool(self.lib.dppo_small_update_supported(C.byref(desc)))

    def small_update(self, desc, params, grads, exp_avg, exp_avg_sq, obs, actions, old_logp, adv, returns, adv_stats, idx, rows, steps,
                     hyper, step_consts, losses, grad_norm_out=None):
        """All `steps` optimiser steps of a learn() in one cluster launch (default 64-wide network; dppo_small_update)."""
        self._check(self.lib.dppo_small_update(self.h, C.byref(desc), _ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq),
                                               _ptr(obs), _ptr(actions), _ptr(old_logp), _ptr(adv), _ptr(returns), _ptr(adv_stats),
                                               _ptr(idx), C.c_int64(rows), C.c_int(steps), C.byref(hyper), _ptr(step_consts),
                                               _ptr(losses), _ptr(grad_norm_out), _stream()), "dppo_small_update")
        self.launches += 1

    # ---- device-resident vector environments -----------------------------------------------------
    def env_reset(self, desc, state, mask=None):
        self._check(self.lib.dppo_env_reset(self.h, C.byref(desc), C.byref(state), _ptr(mask), _stream()), "dppo_env_reset")

    def env_step(self, desc, state, actions, t, auto_reset, obs, next_obs, buf_actions, rewards, terminations, truncations,
                 done_return=None, raw_rewards=None):
        self._check(self.lib.dppo_env_step(self.h, C.byref(desc), C.byref(state), _ptr(actions), C.c_int(t), C.c_int(int(auto_reset)),
                                           _ptr(obs), _ptr(next_obs), _ptr(buf_actions), _ptr(rewards), _ptr(terminations),
                                           _ptr(truncations), _ptr(done_return), _ptr(raw_rewards), _stream()), "dppo_env_step")

    def episode_stats(self, rewards, terminations, truncations, ep_return, ep_len, window, out_returns, out_lengths, out_n, finished, ws):
        """Device-side Ticker bookkeeping of one rollout (dppo_episode_stats)."""
        T, N = rewards.shape
        self._check(self.lib.dppo_episode_stats(self.h, _ptr(rewards), _ptr(terminations), _ptr(truncations), C.c_int(T), C.c_int(N),
                                                _ptr(ep_return), _ptr(ep_len), C.c_int(window), _ptr(out_returns), _ptr(out_lengths),
                                                _ptr(out_n), _ptr(finished), _ptr(ws), C.c_int64(ws.numel() * ws.element_size()),
                                                _stream()), "dppo_episode_stats")
        self.launches += 2

    def eval_episodes(self, rewards, terminations, truncations, quota, slot_offset, ep_return, ep_len, recorded, out_returns, out_lengths,
                      remaining):
        """Evaluation bookkeeping of one [T, N] chunk (dppo_eval_episodes)."""
        T, N = rewards.shape
        self._check(self.lib.dppo_eval_episodes(self.h, _ptr(rewards), _ptr(terminations), _ptr(truncations), C.c_int(T), C.c_int(N),
                                                _ptr(quota), _ptr(slot_offset), _ptr(ep_return), _ptr(ep_len), _ptr(recorded),
                                                _ptr(out_returns), _ptr(out_lengths), _ptr(remaining), _stream()), "dppo_eval_episodes")

    def episode_stats_workspace_bytes(self, T, N):
        return int(self.lib.dppo_episode_stats_workspace_bytes(C.c_int(T), C.c_int(N)))

    # ---- recurrent actor-critic (recurrent_ppo.py) -----------------------------------------------
    def rnn_workspace_bytes(self, desc, T, N, M, training):
        return int(self.lib.dppo_rnn_workspace_bytes(C.byref(desc), C.c_int(T), C.c_int(N), C.c_int64(M), C.c_int(int(training))))

    def rnn_forward(self, desc, params, obs, prev_dones, hx0, T, N, heads, logits, values, hx_out, ws):
        self._check(self.lib.dppo_rnn_forward(self.h, C.byref(desc), _ptr(params), _ptr(obs), _ptr(prev_dones), _ptr(hx0),
                                              C.c_int(T), C.c_int(N), C.c_int(heads), _ptr(logits), _ptr(values), _ptr(hx_out),
                                              _ptr(ws), C.c_int64(ws.numel() * ws.element_size()), _stream()), "dppo_rnn_forward")

    def rnn_grad_minibatch(self, desc, params, grads, obs, prev_dones, hx0, T, N, actions, old_logp, adv, returns, adv_stats, idx, M,
                           hyper, losses, ws):
        self._check(self.lib.dppo_rnn_grad_minibatch(self.h, C.byref(desc), _ptr(params), _ptr(grads), _ptr(obs), _ptr(prev_dones),
                                                     _ptr(hx0), C.c_int(T), C.c_int(N), _ptr(actions), _ptr(old_logp), _ptr(adv),
                                                     _ptr(returns), _ptr(adv_stats), _ptr(idx), C.c_int64(M), C.byref(hyper),
                                                     _ptr(losses), _ptr(ws), C.c_int64(ws.numel() * ws.element_size()), _stream()),
                    "dppo_rnn_grad_minibatch")

    def grad_sumsq_bytes(self, n):
        return int(self.lib.dppo_grad_sumsq_bytes(self.h, C.c_int64(n)))

    def clip_adam_workspace_bytes(self, n):
        return int(self.lib.dppo_clip_adam_workspace_bytes(C.c_int64(n)))

    def clip_adam_step(self, params, grads, exp_avg, exp_avg_sq, hyper, ws, grad_norm_out=None):
        self._check(self.lib.dppo_clip_adam_step(self.h, _ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq),
                                                 C.c_int64(params.numel()), C.byref(hyper), _ptr(grad_norm_out), _ptr(ws),
                                                 C.c_int64(ws.numel() * ws.element_size()), _stream()), "dppo_clip_adam_step")
        self.launches += 2

    # ---- device permutation generator / shard filter ------------------------------------------
    def permutation_device(self, seed, counter, n, out):
        """out[0..n) (int32, device) = keyed-bijection permutation of [0, n) (dppo_permutation_device)."""
        self._check(self.lib.dppo_permutation_device(self.h, C.c_uint64(seed & (2 ** 64 - 1)), C.c_uint64(counter), C.c_int64(n),
                                                     _ptr(out), _stream()), "dppo_permutation_device")
        self.launches += 1
        return out

    def perm_shard_filter(self, perm, B_global, n_global_envs, env_lo, n_local, MB, M_pad, idx_out, counts, overflow):
        self._check(self.lib.dppo_perm_shard_filter(self.h, _ptr(perm), C.c_int64(B_global), C.c_int(n_global_envs), C.c_int(env_lo),
                                                    C.c_int(n_local), C.c_int(MB), C.c_int64(M_pad), _ptr(idx_out), _ptr(counts),
                                                    _ptr(overflow), _stream()), "dppo_perm_shard_filter")
        self.launches += 1

    # ---- standalone pieces for custom networks ------------------------------------------------
    def gather_rows(self, src, idx, out=None):
        rows = idx.numel()
        row_floats = src[0].numel() if src.dim() > 1 else 1
        out = torch.empty((rows,) + tuple(src.shape[1:]), dtype=torch.float32, device=src.device) if out is None else out
        self._check(self.lib.dppo_gather_rows_f32(self.h, _ptr(src), _ptr(idx), _ptr(out), C.c_int64(rows),
                                                  C.c_int(row_floats), _stream()), "dppo_gather_rows_f32")
        self.launches += 1
        return out

    def ppo_loss_workspace_bytes(self, M, A):
        return int(self.lib.dppo_ppo_loss_workspace_bytes(C.c_int64(M), C.c_int(A)))

    def ppo_loss_discrete(self, logits, values, actions_i32, old_logp, adv, returns, hyper, losses, dlogits, dvalues, ws):
        M, A = logits.shape
        self._check(self.lib.dppo_ppo_loss_discrete(self.h, _ptr(logits), _ptr(values), _ptr(actions_i32), _ptr(old_logp),
                                                    _ptr(adv), _ptr(returns), C.c_int64(M), C.c_int(A), C.byref(hyper),
                                                    _ptr(losses), _ptr(dlogits), _ptr(dvalues), _ptr(ws),
                                                    C.c_int64(ws.numel() * ws.element_size()), _stream()), "dppo_ppo_loss_discrete")
        self.launches += 2

    def ppo_loss_gaussian(self, mean, log_std, values, actions, old_logp, adv, returns, hyper, losses, dmean, dlog_std,
                          dvalues, ws, log_std_row_stride=0):
        M, A = mean.shape
        self._check(self.lib.dppo_ppo_loss_gaussian(self.h, _ptr(mean), _ptr(log_std), C.c_int64(log_std_row_stride),
                                                    _ptr(values), _ptr(actions),
                                                    _ptr(old_logp), _ptr(adv), _ptr(returns), C.c_int64(M), C.c_int(A),
                                                    C.byref(hyper), _ptr(losses), _ptr(dmean), _ptr(dlog_std), _ptr(dvalues),
                                                    _ptr(ws), C.c_int64(ws.numel() * ws.element_size()), _stream()),
                    "dppo_ppo_loss_gaussian")
        self.launches += 2

    def tc_linear(self, epi, A, W, transpose, bias=None, Hact=None, colsum=False, out=None, ws=None, prepared=False):
        """C = epi(A op(W)) on the tensor cores (dppo_tc_linear_f32); returns (C, colsum partials or None).
        ws + prepared=True re-uses the weight images an earlier call left in ws (kernel-only timing)."""
        M, K = A.shape
        N = W.shape[1] if transpose else W.shape[0]
        Cm = torch.empty(M, N, device=A.device, dtype=torch.float32) if out is None else out
        parts = self.lib.dppo_tc_colsum_parts(self.h, C.c_int64(M), C.c_int(N))
        cs = torch.zeros(parts, N, device=A.device, dtype=torch.float32) if colsum else None
        if ws is None:
            ws = torch.empty(self.lib.dppo_tc_linear_workspace_bytes(C.c_int(N), C.c_int(K)), device=A.device, dtype=torch.uint8)
        self._check(self.lib.dppo_tc_linear_f32(self.h, C.c_int(epi), _ptr(A), C.c_int64(M), C.c_int(K), _ptr(W), C.c_int(N),
                                                C.c_int(int(transpose)), _ptr(bias), _ptr(Hact), _ptr(Cm), _ptr(cs), _ptr(ws),
                                                C.c_int64(ws.numel()), C.c_int(int(prepared)), _stream()),
                    "dppo_tc_linear_f32")
        self.launches += 2
        return Cm, cs

    def tc_wgrad(self, Dm, Hm):
        """dW = Dm^T Hm on the tensor cores (dppo_tc_wgrad_f32)."""
        M, N1 = Dm.shape
        N2 = Hm.shape[1]
        dW = torch.empty(N1, N2, device=Dm.device, dtype=torch.float32)
        ws = torch.empty(self.lib.dppo_tc_wgrad_workspace_bytes(self.h, C.c_int64(M), C.c_int(N1), C.c_int(N2)), device=Dm.device,
                         dtype=torch.uint8)
        self._check(self.lib.dppo_tc_wgrad_f32(self.h, _ptr(Dm), _ptr(Hm), C.c_int64(M), C.c_int(N1), C.c_int(N2), _ptr(dW), _ptr(ws),
                                               C.c_int64(ws.numel()), _stream()), "dppo_tc_wgrad_f32")
        self.launches += 2
        return dW

    def mma_probe(self, pair, bf16, n, iters):
        """SM cycles per tcgen05.mma (shared-memory operands) measured on every SM; returns (cycles tensor, iters)."""
        out = torch.zeros(self.sm_count, dtype=torch.int64, device="cuda")
        g = C.c_int()
        self._check(self.lib.dppo_tc_mma_probe(self.h, C.c_int(pair), C.c_int(bf16), C.c_int(n), C.c_int(iters), _ptr(out), C.byref(g),
                                               _stream()), "dppo_tc_mma_probe")
        self.launches += 1
        torch.cuda.synchronize()
        o = out[:g.value]
        return o[o > 0].float() / iters

    # ---- data-parallel exchange (dp.cu) --------------------------------------------------------
    def dp_create(self, world, rank, n_floats):
        h = C.c_void_p()
        self._check(self.lib.dppo_dp_create(self.h, C.c_int(world), C.c_int(rank), C.c_int64(n_floats), C.byref(h)), "dppo_dp_create")
        return h

    def dp_handle(self, dp) -> bytes:
        buf = C.create_string_buffer(self.lib.dppo_dp_handle_bytes())
        self.lib.dppo_dp_handle(dp, buf)
        return buf.raw

    def dp_connect(self, dp, all_handles: bytes):
        self._check(self.lib.dppo_dp_connect(self.h, dp, C.c_char_p(all_handles)), "dppo_dp_connect")

    def dp_slot(self, dp, seq) -> int:
        return int(self.lib.dppo_dp_slot(dp, C.c_int64(seq)))

    def dp_zero_slot(self, dp, seq):
        self._check(self.lib.dppo_dp_zero_slot(self.h, dp, C.c_int64(seq), _stream()), "dppo_dp_zero_slot")

    def dp_workspace_bytes(self, n):
        return int(self.lib.dppo_dp_workspace_bytes(C.c_int64(n)))

    def dp_status(self, dp) -> int:
        """0: fine; 1 + q: an exchange kernel gave up waiting for rank q (crashed / desynchronised peer).  No synchronisation."""
        return int(self.lib.dppo_dp_status(dp))

    def dp_allreduce_clip_adam(self, dp, seq, params, grads_out, exp_avg, exp_avg_sq, hyper, losses_out, ws, grad_norm_out=None):
        self._check(self.lib.dppo_dp_allreduce_clip_adam(self.h, dp, C.c_int64(seq), _ptr(params), _ptr(grads_out), _ptr(exp_avg), _ptr(exp_avg_sq),
                                                         C.byref(hyper), _ptr(losses_out), _ptr(grad_norm_out), _ptr(ws),
                                                         C.c_int64(ws.numel() * ws.element_size()), _stream()),
                    "dppo_dp_allreduce_clip_adam")
        self.launches += 2

    def dp_destroy(self, dp):
        self.lib.dppo_dp_destroy(dp)

    def fma_peak(self, sink, iters):
        b, t = C.c_int(), C.c_int()
        self._check(self.lib.dppo_fma_peak_kernel(self.h, _ptr(sink), C.c_int64(iters), C.byref(b), C.byref(t), _stream()),
                    "dppo_fma_peak_kernel")
        self.launches += 1
        return b.value, t.value


_contexts: dict[int, Context] = {}


def get_context(device: int | None = None) -> Context:
    dev = torch.cuda.current_device() if (device is None and torch.cuda.is_available()) else device
    if dev not in _contexts:
        _contexts[dev] = Context(dev)
    return _contexts[dev]
