"""diamond — B200-native drop-in for the hot path of Diamond PPO (same import surface as the
reference package: diamond/__init__.py:1-3).  Submodules are imported on first use."""
__all__ = ["PPO", "PPOConfig", "ContinuousPPO", "ContinuousPPOConfig", "RecurrentPPO", "RecurrentPPOConfig",
           "RecurrentContinuousPPO", "RecurrentContinuousPPOConfig"]

_WHERE = {
    "PPO": "agents", "ContinuousPPO": "agents", "RecurrentPPO": "recurrent", "RecurrentContinuousPPO": "recurrent",
    "PPOConfig": "config", "ContinuousPPOConfig": "config", "RecurrentPPOConfig": "config", "RecurrentContinuousPPOConfig": "config",
}


def __getattr__(name):
    if name in _WHERE:
        import importlib
        return getattr(importlib.import_module(f".{_WHERE[name]}", __name__), name)
    raise AttributeError(name)
