"""TEST INFRASTRUCTURE ONLY - ctypes wrapper of the host emulation of the tree-search kernels (tests/emu/mcts_emu.cpp).

EmuMCTS takes an EmuBatch of tests/emu/emu.py: mcts_emu.cpp is compiled on top of the same hexb_emu.cpp, so its idea of an emulator
handle is the step emulator's. The tree is a host uint8 array in the layout of hex_gym_env_b200/csrc/hexb_mcts.cuh."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "libhexb_mcts_emu.so")
    srcs = [os.path.join(_HERE, f) for f in ("mcts_emu.cpp", "hexb_emu.cpp")] + [
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
        L.emu_mcts_tree_bytes.restype = ctypes.c_longlong
        L.emu_mcts_tree_bytes.argtypes = [ctypes.c_int, ctypes.c_longlong, ctypes.c_int]
        L.emu_mcts.argtypes = [vp, ctypes.c_int, vp, ctypes.c_longlong, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_longlong,
                               vp, ctypes.c_int, ctypes.c_int] + [vp] * 9
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class EmuMCTS(object):
    """hexb_mcts_* on an EmuBatch, with the method surface of hex_gym_env_b200.MCTS (numpy in and out)."""

    def __init__(self, batch, max_nodes, c_puct=1.25, fpu=0.0):
        self.batch, self.max_nodes, self.c_puct, self.fpu = batch, int(max_nodes), float(c_puct), float(fpu)
        self.tree = np.zeros(int(lib().emu_mcts_tree_bytes(batch.N, batch.G, self.max_nodes)), np.uint8)

    def _call(self, op, **kw):
        a = dict(max_nodes=self.max_nodes, c_puct=self.c_puct, fpu=self.fpu, first_playout=0, root_mask=None, sims=0, playouts=0)
        a.update(kw)
        ptrs = [_p(kw.get(k)) for k in ("leaf_obs", "leaf_mask", "pending", "priors", "values", "visits", "q", "value", "nodes_used")]
        lib().emu_mcts(self.batch._h, op, _p(self.tree), self.tree.size, a["max_nodes"], a["c_puct"], a["fpu"], int(a["first_playout"]),
                       _p(a["root_mask"]), int(a["sims"]), int(a["playouts"]), *ptrs)

    def reset(self, root_mask=None, first_playout=0):
        rm = None if root_mask is None else np.ascontiguousarray(root_mask, np.uint8)
        self._call(0, root_mask=rm, first_playout=first_playout)

    def search(self, num_simulations, playouts_per_leaf):
        self._call(1, sims=num_simulations, playouts=playouts_per_leaf)

    def select(self):
        G, N, C = self.batch.G, self.batch.N, self.batch.C
        obs, mask, pending = np.zeros((G, N, N), np.int8), np.zeros((G, C), np.uint8), np.zeros(G, np.uint8)
        self._call(2, leaf_obs=obs, leaf_mask=mask, pending=pending)
        return obs, mask, pending

    def expand(self, priors, values):
        self._call(3, priors=np.ascontiguousarray(priors, np.float32), values=np.ascontiguousarray(values, np.float32))

    def root(self):
        G, C = self.batch.G, self.batch.C
        out = dict(visits=np.zeros((G, C), np.int32), q=np.zeros((G, C), np.float32), value=np.zeros(G, np.float32),
                   nodes_used=np.zeros(G, np.int32))
        self._call(4, **out)
        return out["visits"], out["q"], out["value"], out["nodes_used"]
