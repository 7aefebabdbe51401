"""Hyper-parameter dataclasses.  PPOConfig, ContinuousPPOConfig and RecurrentPPOConfig are field-for-field
identical to the reference's so that user code and subclasses (notebook cell 9) keep working: diamond/ppo.py:15-37,
diamond/continuous_ppo.py:15-37, diamond/recurrent_ppo.py:15-38.  RecurrentContinuousPPOConfig (the Gaussian-policy
recurrent agent, which the reference does not have) has RecurrentPPOConfig's fields and defaults, as ContinuousPPOConfig
has PPOConfig's.  B200-specific knobs are keyword arguments of the agents, never config fields."""
from dataclasses import dataclass


@dataclass
class _CommonConfig:
    total_steps: int = 1_000_000        # env steps for the whole run
    rollout_steps: int = 64             # T: vectorised steps per rollout
    num_envs: int = 16                  # N: parallel envs
    lr: float = 3e-4                    # Adam learning rate
    adam_eps: float = 1e-5              # Adam epsilon
    decay_lr: bool = False              # LinearLR to 5 % over the run
    gamma: float = 0.99                 # discount
    gae_lambda: float = 0.95            # GAE lambda
    num_epochs: int = 4                 # E: passes over the rollout per update
    num_minibatches: int = 8            # MB: optimiser steps per epoch
    ppo_clip: float = 0.2               # ratio clip epsilon
    value_loss_weight: float = 1.0      # value-loss coefficient
    entropy_beta: float = 0.01          # entropy bonus coefficient
    advantage_norm: bool = True         # batch-normalise advantages
    grad_norm_clip: float = 0.5         # global grad-norm clip
    network_hidden_dim: int = 64        # H of the default MLP


@dataclass
class _TailConfig:
    cuda: bool = False                  # kept for API compatibility; this package always runs on the GPU
    seed: int | None = 42               # seeds numpy + torch
    checkpoint: bool = False            # periodic checkpoints
    save_interval: float = 600          # seconds between checkpoints
    verbose: bool = True                # Ticker console output


@dataclass
class PPOConfig(_TailConfig, _CommonConfig):
    pass


@dataclass
class ContinuousPPOConfig(_TailConfig, _CommonConfig):
    pass


@dataclass
class _RecurrentExtra:
    gru_hidden_dim: int = 16            # Hg


@dataclass
class RecurrentPPOConfig(_TailConfig, _RecurrentExtra, _CommonConfig):
    # recurrent defaults differ (recurrent_ppo.py:18-19,25-27)
    rollout_steps: int = 32
    num_envs: int = 32
    num_epochs: int = 10
    num_minibatches: int = 1
    ppo_clip: float = 0.15


@dataclass
class RecurrentContinuousPPOConfig(_TailConfig, _RecurrentExtra, _CommonConfig):
    # RecurrentPPOConfig's defaults
    rollout_steps: int = 32
    num_envs: int = 32
    num_epochs: int = 10
    num_minibatches: int = 1
    ppo_clip: float = 0.15
