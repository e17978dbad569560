"""ctypes binding of libhexb.so (the C ABI declared in include/hexb.h).

The library is built in-tree by :func:`build` (``nvcc -gencode arch=compute_100a,code=sm_100a``). There is no CPU
implementation behind this module: if the shared library cannot be built or loaded, importing a simulator class fails
with a RuntimeError.
"""
import ctypes
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libhexb.so")
HEADER = os.path.join(_HERE, "include", "hexb.h")                           # the copy that ships inside the package
ROOT_HEADER = os.path.join(os.path.dirname(_HERE), "include", "hexb.h")      # the repository's canonical include/hexb.h
BUILD_DIR = os.path.join(_HERE, "build")
BOARD_SIZES = list(range(3, 20))
_DEVICE_HEADERS = ["hexb_core.cuh", "hexb_phases.cuh", "hexb_views.cuh", "hexb_search.cuh", "hexb_mcts.cuh", "hexb_step.cuh", "hexb_host.h"]
SOURCES = [os.path.join(_CSRC, f) for f in ["hexb_kernels.cu", "hexb_step_inst.cu", "hexb_hostpack.cpp"] + _DEVICE_HEADERS] + [HEADER]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def _sync_header():
    """include/hexb.h at the repository root is the canonical header; the package carries a copy so that an installed package
    (pip install ., wheel) can rebuild without the repository around it. Keep the copy identical when both exist."""
    if os.path.isfile(ROOT_HEADER):
        with open(ROOT_HEADER, "rb") as f:
            want = f.read()
        have = None
        if os.path.isfile(HEADER):
            with open(HEADER, "rb") as f:
                have = f.read()
        if have != want:
            os.makedirs(os.path.dirname(HEADER), exist_ok=True)
            with open(HEADER, "wb") as f:
                f.write(want)


def _mtime(path):
    return os.path.getmtime(path) if os.path.exists(path) else None


def _run(cmd):
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        raise RuntimeError("building libhexb.so failed:\n%s\n%s" % (" ".join(cmd), proc.stdout))
    return proc.stdout


def build(force=False, verbose=False, jobs=None):
    """Compile libhexb.so for sm_100a if it is missing or older than its sources. Returns the library path.

    One object per board size (csrc/hexb_step_inst.cu with -DHEXB_INST_N=n: every instantiation of the step kernels for that N),
    hexb_kernels.cu (C ABI + size-independent kernels) and hexb_hostpack.cpp (host only), compiled in parallel and linked."""
    def stale():
        if not os.path.exists(LIB_PATH):
            return True
        if not os.path.isfile(ROOT_HEADER):
            return False      # an installed package (no repository around it): file times say nothing there, the shipped library is used
        have = [s for s in SOURCES if os.path.exists(s)]
        return any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in have)

    try:
        _sync_header()
    except OSError:
        pass                                                # read-only install: use what is there
    if force or stale():
        import fcntl
        from concurrent.futures import ThreadPoolExecutor
        with open(LIB_PATH + ".lock", "w") as lock:     # one builder at a time (torchrun starts several ranks at once)
            fcntl.flock(lock, fcntl.LOCK_EX)
            if force or stale():                        # another rank may have built it while we waited
                missing = [s for s in SOURCES if not os.path.exists(s)]
                if missing:
                    raise RuntimeError("cannot build libhexb.so: missing sources %s" % (missing,))
                os.makedirs(BUILD_DIR, exist_ok=True)
                hdrs = [os.path.join(_CSRC, h) for h in _DEVICE_HEADERS] + [HEADER]
                newest_hdr = max(os.path.getmtime(h) for h in hdrs)
                extra = ["-Xptxas", "-v"] if verbose else []
                units = []      # (object, command)
                inst = os.path.join(_CSRC, "hexb_step_inst.cu")
                for n in BOARD_SIZES:
                    units.append((os.path.join(BUILD_DIR, "step_%d.o" % n), inst,
                                  [_nvcc()] + NVCC_FLAGS + extra + ["-DHEXB_INST_N=%d" % n, "-c", inst]))
                abi = os.path.join(_CSRC, "hexb_kernels.cu")
                units.append((os.path.join(BUILD_DIR, "abi.o"), abi, [_nvcc()] + NVCC_FLAGS + extra + ["-c", abi]))
                hp = os.path.join(_CSRC, "hexb_hostpack.cpp")
                units.append((os.path.join(BUILD_DIR, "hostpack.o"), hp,
                              ["g++", "-O3", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-pthread", "-c", hp]))
                todo = []
                for obj, src, cmd in units:
                    mt = _mtime(obj)
                    if force or mt is None or mt < max(os.path.getmtime(src), newest_hdr):
                        todo.append(cmd + ["-o", obj])
                workers = jobs or max(1, min(len(todo), len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else 4))
                with ThreadPoolExecutor(max_workers=workers) as ex:
                    logs = list(ex.map(_run, todo))
                tmp = "%s.%d.tmp" % (LIB_PATH, os.getpid())
                try:
                    _run([_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-o", tmp] + [u[0] for u in units] + ["-lpthread"])
                except RuntimeError:
                    if os.path.exists(tmp):
                        os.remove(tmp)
                    raise
                os.replace(tmp, LIB_PATH)               # atomic: a concurrent loader never sees a half-written library
                if verbose:
                    print("\n".join(logs))
    return LIB_PATH


class HexbConfig(ctypes.Structure):
    _fields_ = [("board_size", ctypes.c_int32), ("variant", ctypes.c_int32), ("num_games", ctypes.c_int64),
                ("game_offset", ctypes.c_int64), ("seed", ctypes.c_uint64), ("agent_mode", ctypes.c_int32),
                ("opponent_first", ctypes.c_int32), ("auto_reset", ctypes.c_int32), ("eval_state", ctypes.c_int32),
                ("raw", ctypes.c_int32), ("device", ctypes.c_int32), ("manual_opponent", ctypes.c_int32),
                ("pool_size", ctypes.c_int32), ("obs_dtype", ctypes.c_int32)]


# every symbol include/hexb.h declares: name -> (restype, argtypes)
_vp, _i32, _sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t
_cfgp = ctypes.POINTER(HexbConfig)
SYMBOLS = {
    "hexb_version": (_i32, []),
    "hexb_strerror": (ctypes.c_char_p, [_i32]),
    "hexb_last_cuda_error": (_i32, []),
    "hexb_state_bytes": (_sz, [_cfgp]),
    "hexb_create": (_i32, [_cfgp, _vp, _sz, _vp, ctypes.POINTER(_vp)]),
    "hexb_destroy": (_i32, [_vp]),
    "hexb_get_config": (_i32, [_vp, _cfgp]),
    "hexb_reset": (_i32, [_vp] * 6),
    "hexb_step": (_i32, [_vp] * 10),
    "hexb_host_workspace_bytes": (_sz, [_cfgp]),
    "hexb_step_host": (_i32, [_vp] * 8),
    "hexb_step_host_begin": (_i32, [_vp] * 8),
    "hexb_step_host_end": (_i32, [_vp]),
    "hexb_host_packed_bytes": (_sz, [_cfgp]),
    "hexb_step_host_packed": (_i32, [_vp] * 9),
    "hexb_host_threads": (_i32, []),
    "hexb_mem_alloc": (_i32, [_i32, _sz, _i32, ctypes.POINTER(_vp), ctypes.POINTER(_i32)]),
    "hexb_mem_free": (_i32, [_vp]),
    "hexb_set_host_transport": (_i32, [_vp, ctypes.c_double]),
    "hexb_get_host_transport": (_i32, [_vp, ctypes.POINTER(ctypes.c_double)]),
    "hexb_set_launch_form": (_i32, [_vp, _i32]),
    "hexb_gae": (_i32, [_vp, _vp, _vp, _i32, ctypes.c_int64, ctypes.c_double, ctypes.c_double, _vp, _vp, _i32, _vp]),
    "hexb_ply": (_i32, [_vp] * 4),
    "hexb_encode": (_i32, [_vp, _i32, _vp, _vp, _vp]),
    "hexb_sample_actions": (_i32, [_vp, _i32, _vp, _vp, _vp]),
    "hexb_export_state": (_i32, [_vp] * 10),
    "hexb_import_boards": (_i32, [_vp] * 5),
    "hexb_import_labels": (_i32, [_vp] * 6),
    "hexb_stats": (_i32, [_vp] * 3),
    "hexb_rollout": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hexb_set_opponent_buffers": (_i32, [_vp, _vp, _vp]),
    "hexb_set_info_buffers": (_i32, [_vp, _vp, _vp]),
    "hexb_set_eval": (_i32, [_vp, _i32, _vp, _vp]),
    "hexb_set_opponent_eps": (_i32, [_vp, ctypes.c_double]),
    "hexb_half_step": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "hexb_masked_sample": (_i32, [_vp, _vp, _vp, ctypes.c_int64, _i32, _vp, _vp, _vp, _i32, _vp]),
    "hexb_copy_games": (_i32, [_vp, _vp, _vp, _vp, ctypes.c_int64, _vp]),
    "hexb_playouts": (_i32, [_vp, _i32, ctypes.c_int64, _vp, _vp, _vp]),
    "hexb_playouts_policy": (_i32, [_vp, _i32, ctypes.c_int64, _i32, _vp, _vp, _vp]),
    "hexb_mcts_tree_bytes": (_i32, [_vp, _i32, ctypes.POINTER(_sz)]),
    "hexb_mcts_init": (_i32, [_vp, _vp, _sz, _i32, ctypes.c_double, ctypes.c_double, ctypes.c_int64, _vp, _vp]),
    "hexb_mcts_search": (_i32, [_vp, _vp, _sz, _i32, _i32, _vp]),
    "hexb_mcts_search_policy": (_i32, [_vp, _vp, _sz, _i32, _i32, _i32, _vp]),
    "hexb_mcts_select": (_i32, [_vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "hexb_mcts_expand": (_i32, [_vp, _vp, _sz, _vp, _vp, _vp]),
    "hexb_mcts_root": (_i32, [_vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp]),
    "hexb_mcts_advance": (_i32, [_vp, _vp, _sz, ctypes.c_int64, _vp, _vp]),
}

_LIB = None


def lib():
    """The loaded library. Raises RuntimeError (never falls back) if it cannot be built or loaded."""
    global _LIB
    if _LIB is None:
        try:
            # HEXB_LIB: load this build of the same CUDA library instead (kernel-tuning experiments, e.g. other CTA shapes)
            path = os.environ.get("HEXB_LIB") or build()
            L = ctypes.CDLL(path)
        except (OSError, RuntimeError) as exc:
            raise RuntimeError("hex_gym_env_b200: the CUDA library libhexb.so is required and could not be loaded "
                               "(%s). There is no CPU fallback." % (exc,))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _LIB = L
    return _LIB


class HexbError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        L = lib()
        msg = L.hexb_strerror(rc).decode()
        if rc == -2:
            msg += " (cudaError %d)" % L.hexb_last_cuda_error()
        raise HexbError("libhexb: %s" % msg)


class DeviceBuffer(object):
    """`nbytes` of device memory from hexb_mem_alloc (compressible if asked and granted), exposed through
    __cuda_array_interface__ so that torch.as_tensor(buf, device=...) aliases it; freed when the last tensor over it is gone."""

    def __init__(self, nbytes, device, compressible=True):
        L = lib()
        p, got = ctypes.c_void_p(), ctypes.c_int32(0)
        rc = L.hexb_mem_alloc(int(device), int(nbytes), 1 if compressible else 0, ctypes.byref(p), ctypes.byref(got))
        if rc != 0 or not p.value:
            raise RuntimeError("hexb_mem_alloc(%d bytes) failed: %s" % (nbytes, L.hexb_strerror(rc).decode()))
        self.ptr, self.nbytes, self.compressed, self._lib = int(p.value), int(nbytes), bool(got.value), L
        self.__cuda_array_interface__ = {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 2}

    def __del__(self):
        try:
            if getattr(self, "ptr", 0):
                self._lib.hexb_mem_free(ctypes.c_void_p(self.ptr))
                self.ptr = 0
        except Exception:
            pass
