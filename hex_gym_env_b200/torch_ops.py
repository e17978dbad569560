"""torch.ops.hexb.* - the C ABI of libhexb.so registered as PyTorch operators (csrc/hexb_torch.cpp).

The operators are the same thin layer as the ctypes binding (_native.py), in C++: tensor checks, the current CUDA stream,
raw pointers into the extern "C" entry points. Use them when the step has to appear as an operator (torch.library schemas with
mutable outputs, CUDA-graph capture through torch, C++ callers of libtorch); HexBatch itself stays on ctypes, which needs no
torch headers to build.

    from hex_gym_env_b200 import HexBatch, torch_ops
    ops = torch_ops.load()                                  # builds libhexb_torch.so in-tree on first use
    env = HexBatch(11, 1 << 20, variant=1, agent_mode=2)
    ops.reset(env.handle, None, None, obs, mask)
    ops.step(env.handle, None, None, obs, mask, reward, done, None, None)
    ops.copy_games(children.handle, env.handle, roots, None, roots.numel())   # children: a raw HexBatch
    ops.playouts(children.handle, 64, 0, None, wins)
    ops.mcts_init(env.handle, tree, 801, 1.25, 0.0, 0, None)                    # tree: uint8[hexb_mcts_tree_bytes] (mcts.MCTS)
    ops.mcts_search(env.handle, tree, 800, 8)
    ops.mcts_search(env.handle, tree, 800, 8, policy=1)                      # bridge playouts (PLAYOUT_BRIDGE)

There is no CPU implementation behind the operators: they raise unless their tensors live on the handle's CUDA device.
"""
import os
import shutil
import subprocess

from . import _native

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_HERE, "csrc", "hexb_torch.cpp")
LIB_PATH = os.path.join(_HERE, "libhexb_torch.so")
_LOADED = False


def build(force=False):
    """Compile libhexb_torch.so (host C++ only: the kernels stay in libhexb.so, which it links with rpath $ORIGIN)."""
    import torch
    from torch.utils import cpp_extension as ce
    base = _native.build()
    deps = [SRC, _native.HEADER]

    def stale():
        return (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(d) > os.path.getmtime(LIB_PATH) for d in deps)

    if force or stale():
        import fcntl
        with open(LIB_PATH + ".lock", "w") as lock:
            fcntl.flock(lock, fcntl.LOCK_EX)
            if force or stale():
                cuda_home = os.environ.get("CUDA_HOME") or os.path.dirname(os.path.dirname(shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"))
                tmp = "%s.%d.tmp" % (LIB_PATH, os.getpid())
                cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI)]
                cmd += ["-I" + p for p in ce.include_paths()] + ["-I" + os.path.join(cuda_home, "include")]
                cmd += [SRC, "-o", tmp, "-L" + os.path.dirname(base), "-l:libhexb.so", "-Wl,-rpath,$ORIGIN"]
                cmd += ["-L" + p for p in ce.library_paths()] + ["-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda", "-ltorch"]
                cmd += ["-L" + os.path.join(cuda_home, "lib64"), "-lcudart"]
                proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                if proc.returncode != 0:
                    if os.path.exists(tmp):
                        os.remove(tmp)
                    raise RuntimeError("building libhexb_torch.so failed:\n%s\n%s" % (" ".join(cmd), proc.stdout))
                os.replace(tmp, LIB_PATH)
    return LIB_PATH


def load():
    """Register the operators (once) and return the torch.ops.hexb namespace."""
    global _LOADED
    import torch
    if not _LOADED:
        torch.ops.load_library(build())
        _LOADED = True
    return torch.ops.hexb
