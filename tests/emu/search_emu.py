"""TEST INFRASTRUCTURE ONLY - ctypes wrapper of the host emulation of the tree-search kernels (tests/emu/search_emu.cpp).

The functions take EmuBatch objects of tests/emu/emu.py: search_emu.cpp is compiled on top of the same hexb_emu.cpp, so its idea of
an emulator handle is the step emulator's."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "libhexb_search_emu.so")
    srcs = [os.path.join(_HERE, f) for f in ("search_emu.cpp", "hexb_emu.cpp")] + [
        os.path.join(_ROOT, "hex_gym_env_b200", "csrc", f) for f in ("hexb_core.cuh", "hexb_phases.cuh", "hexb_views.cuh", "hexb_search.cuh")]
    if force or not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-Wall", "-Wno-unknown-pragmas",
                               "-o", so, srcs[0]])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        vp = ctypes.c_void_p
        L.emu_copy_games.argtypes = [vp, vp, vp, vp, ctypes.c_longlong]
        L.emu_playouts.argtypes = [vp, ctypes.c_int, ctypes.c_longlong, vp, vp]
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def copy_games(dst, src, src_index=None, dst_index=None, count=None):
    """hexb_copy_games between two EmuBatch objects (dst raw, same N and variant)."""
    si = None if src_index is None else np.ascontiguousarray(src_index, np.int64)
    di = None if dst_index is None else np.ascontiguousarray(dst_index, np.int64)
    if count is None:
        count = len(si) if si is not None else (len(di) if di is not None else min(dst.G, src.G))
    lib().emu_copy_games(dst._h, src._h, _p(si), _p(di), int(count))


def playouts(batch, num_playouts, first_playout=0, game_mask=None):
    """hexb_playouts on an EmuBatch: wins i32[G]."""
    wins = np.empty(batch.G, np.int32)
    gm = None if game_mask is None else np.ascontiguousarray(game_mask, np.uint8)
    lib().emu_playouts(batch._h, int(num_playouts), int(first_playout), _p(gm), _p(wins))
    return wins
