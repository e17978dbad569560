"""hex_gym_env_b200 - B200-native batched Hex simulator behind the minihex HexGame / HexEnv / SelfPlayEnv API.

The hot path (stone placement, region-label merging, win check, random opponent, observation + legal-action mask)
runs in hand-written sm_100a CUDA kernels (csrc/) reached through the C ABI of include/hexb.h. Importing this package
does not need a GPU; creating a simulator does, and fails loudly without one (no CPU fallback).
"""
from ._native import HexbError, build, lib  # noqa: F401
from .batch import (AGENT_BLACK, AGENT_RANDOM, AGENT_WHITE, STAT_NAMES, VARIANT_A, VARIANT_B, HexBatch)  # noqa: F401
from .mcts import MCTS  # noqa: F401
from .opponents import OpponentPool, StackedMlpOpponents, evaluate_pool  # noqa: F401

__all__ = ["HexBatch", "HexbError", "build", "lib", "VARIANT_A", "VARIANT_B", "AGENT_BLACK", "AGENT_WHITE", "AGENT_RANDOM",
           "STAT_NAMES", "MCTS", "OpponentPool", "StackedMlpOpponents", "evaluate_pool"]
