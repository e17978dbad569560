"""TEST INFRASTRUCTURE ONLY - ctypes wrapper of the host emulation of the playout kernels of both policies (tests/emu/bridge_emu.cpp):
hexb_playouts_policy and hexb_mcts_search_policy.

The functions take EmuBatch objects of tests/emu/emu.py, and EmuMCTS extends mcts_emu.EmuMCTS with search(S, P, policy): the library
is compiled on top of the same mcts_emu.cpp and hexb_emu.cpp, so its handle and its tree buffer are theirs."""
import ctypes
import os
import subprocess

import numpy as np

from . import mcts_emu

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None
POLICIES = (0, 1)   # PLAYOUT_RANDOM, PLAYOUT_BRIDGE


def build(force=False):
    so = os.path.join(_HERE, "libhexb_bridge_emu.so")
    srcs = [os.path.join(_HERE, f) for f in ("bridge_emu.cpp", "mcts_emu.cpp", "hexb_emu.cpp")] + [
        os.path.join(_ROOT, "hex_gym_env_b200", "csrc", f)
        for f in ("hexb_core.cuh", "hexb_phases.cuh", "hexb_views.cuh", "hexb_search.cuh", "hexb_mcts.cuh")]
    if force or not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-Wall", "-Wno-unknown-pragmas",
                               "-o", so, srcs[0]])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        vp = ctypes.c_void_p
        L.emu_playouts_policy.argtypes = [vp, ctypes.c_int, ctypes.c_longlong, ctypes.c_int, vp, vp]
        L.emu_mcts_search_policy.argtypes = [vp, vp, ctypes.c_longlong, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        _LIB = L
    return _LIB


def _policy(policy):
    if policy not in POLICIES:
        raise ValueError("policy must be 0 (random) or 1 (bridge)")
    return int(policy)


def playouts(batch, num_playouts, first_playout=0, game_mask=None, policy=0):
    """hexb_playouts_policy on an EmuBatch: wins i32[G]."""
    policy = _policy(policy)
    wins = np.empty(batch.G, np.int32)
    gm = None if game_mask is None else np.ascontiguousarray(game_mask, np.uint8)
    lib().emu_playouts_policy(batch._h, int(num_playouts), int(first_playout), policy, mcts_emu._p(gm), mcts_emu._p(wins))
    return wins


class EmuMCTS(mcts_emu.EmuMCTS):
    """mcts_emu.EmuMCTS whose fused search takes a playout policy (hexb_mcts_search_policy)."""

    def search(self, num_simulations, playouts_per_leaf, policy=0):
        policy = _policy(policy)
        lib().emu_mcts_search_policy(self.batch._h, mcts_emu._p(self.tree), self.tree.size, int(num_simulations),
                                     int(playouts_per_leaf), policy)
