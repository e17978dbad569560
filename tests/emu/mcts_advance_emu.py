"""TEST INFRASTRUCTURE ONLY - ctypes wrapper of the host emulation of the tree-reuse kernel (tests/emu/mcts_advance_emu.cpp).

EmuMCTS of mcts_emu.py with advance(): the tree is the same host uint8 array, and the handle the step emulator's (the library is
compiled on top of the same mcts_emu.cpp and hexb_emu.cpp)."""
import ctypes
import os
import subprocess

import numpy as np

from . import mcts_emu

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "libhexb_mcts_advance_emu.so")
    srcs = [os.path.join(_HERE, f) for f in ("mcts_advance_emu.cpp", "mcts_emu.cpp", "hexb_emu.cpp")] + [
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
        L.emu_mcts_advance.argtypes = [vp, vp, ctypes.c_longlong, ctypes.c_longlong, vp]
        _LIB = L
    return _LIB


class EmuMCTS(mcts_emu.EmuMCTS):
    """mcts_emu.EmuMCTS with hexb_mcts_advance (numpy in and out, the method surface of hex_gym_env_b200.MCTS)."""

    def advance(self, root_mask=None, first_playout=0):
        rm = None if root_mask is None else np.ascontiguousarray(root_mask, np.uint8)
        lib().emu_mcts_advance(self.batch._h, mcts_emu._p(self.tree), self.tree.size, int(first_playout), mcts_emu._p(rm))
