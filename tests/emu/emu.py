"""TEST INFRASTRUCTURE ONLY - ctypes wrapper of the host emulator of the CUDA kernels (tests/emu/hexb_emu.cpp).

EmuBatch has the method surface of oracle.hexref.RefBatch, so that tests/parity.py can drive either side. copy_games, playouts and
EmuMCTS emulate hexb_copy_games, hexb_playouts_policy and the hexb_mcts_* calls on EmuBatch handles; EmuMCTS has the method
surface of hex_gym_env_b200.MCTS, and its tree is a host uint8 array in the layout of hex_gym_env_b200/csrc/hexb_mcts.cuh."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None
POLICIES = (0, 1)   # PLAYOUT_RANDOM, PLAYOUT_BRIDGE
MCTS_INIT, MCTS_SEARCH, MCTS_SELECT, MCTS_EXPAND, MCTS_ROOT, MCTS_ADVANCE = range(6)   # op of emu_mcts (csrc/hexb_mcts.cuh)


def build(force=False):
    if os.environ.get("HEXB_EMU_LIB"):      # a prebuilt variant, e.g. the sanitizer build of tools/emu_sanitize.py
        return os.environ["HEXB_EMU_LIB"]
    so = os.path.join(_HERE, "libhexb_emu.so")
    srcs = [os.path.join(_HERE, "hexb_emu.cpp")] + [
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
        vp, i32, i64, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_ulonglong
        L.emu_create.restype = vp
        L.emu_create.argtypes = [i32, i32, i64, i64, u64, i32, i32, i32, i32, i32]
        L.emu_destroy.argtypes = [vp]
        L.emu_reset.argtypes = [vp] * 5
        L.emu_step.argtypes = [vp] * 9
        L.emu_ply.argtypes = [vp] * 3
        L.emu_encode.argtypes = [vp, i32, vp, vp]
        L.emu_sample_actions.argtypes = [vp, i32, vp, vp]
        L.emu_export_state.argtypes = [vp] * 9
        L.emu_import_boards.argtypes = [vp] * 4
        L.emu_stats.argtypes = [vp, vp]
        L.emu_set_manual_opponent.argtypes = [vp, i32, vp, vp]
        L.emu_half_step.argtypes = [vp, i32, vp, vp, vp, vp]
        L.emu_set_eval.argtypes = [vp, i32, vp, i64]
        L.emu_set_opponent_eps.argtypes = [vp, ctypes.c_double]
        L.emu_set_info.argtypes = [vp, vp, vp]
        L.emu_rollout.argtypes = [vp, i32] + [vp] * 6
        L.emu_force_sweep.argtypes = [i32]
        L.emu_import_labels.argtypes = [vp] * 5
        L.emu_philox4x32_10.argtypes = [vp] * 3
        L.emu_draw01.restype = ctypes.c_double
        L.emu_draw01.argtypes = [u64, u64, ctypes.c_uint32]
        L.emu_encode_word.argtypes = [ctypes.c_uint32, i32, vp, vp]
        L.emu_encode_byte.argtypes = [ctypes.c_uint32, i32, vp, vp]
        L.emu_copy_games.argtypes = [vp, vp, vp, vp, i64]
        L.emu_playouts.argtypes = [vp, i32, i64, i32, vp, vp]
        L.emu_mcts_tree_bytes.restype = i64
        L.emu_mcts_tree_bytes.argtypes = [i32, i64, i32]
        L.emu_mcts.argtypes = [vp, i32, vp, i64, i32, ctypes.c_double, ctypes.c_double, i64, vp, i32, i32, i32] + [vp] * 9
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def force_sweep(form):
    """-1: the relabel sweep the device would pick for a small batch; 0: one row per pass; 1: several rows per pass."""
    lib().emu_force_sweep(int(form))


class EmuBatch(object):
    def __init__(self, variant, board_size, num_games, seed=0, game_offset=0, agent_mode=0, opponent_first=False,
                 auto_reset=True, eval_state=False, raw=False, manual_opponent=False, pool_size=0):
        self.N, self.G, self.C = board_size, num_games, board_size * board_size
        self._h = lib().emu_create(board_size, variant, num_games, game_offset, seed, agent_mode, int(opponent_first),
                                   int(auto_reset), int(eval_state), int(raw))
        if not self._h:
            raise ValueError("bad emulator config")
        if manual_opponent:
            self.opp_index = np.full(num_games, -1, np.int32)
            self.to_move = np.full(num_games, 9, np.uint8)
            lib().emu_set_manual_opponent(self._h, pool_size, _p(self.opp_index), _p(self.to_move))

    def set_opponent_eps(self, eps):
        lib().emu_set_opponent_eps(self._h, float(eps))

    def set_eval(self, eval_state):
        if getattr(self, "eval_episode", None) is None:
            self.eval_episode = np.zeros(self.G, np.int32)
        lib().emu_set_eval(self._h, int(bool(eval_state)), _p(self.eval_episode), self.G)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().emu_destroy(self._h)
            self._h = None

    def reset(self, reset_mask=None, open_u=None):
        obs = np.empty((self.G, self.N, self.N), np.int8)
        mask = np.empty((self.G, self.C), np.uint8)
        rm = None if reset_mask is None else np.ascontiguousarray(reset_mask, np.uint8)
        ou = None if open_u is None else np.ascontiguousarray(open_u, np.float64)
        lib().emu_reset(self._h, _p(rm), _p(ou), _p(obs), _p(mask))
        return obs, mask

    def step(self, actions=None, opp_u=None, want_term=False):
        obs = np.empty((self.G, self.N, self.N), np.int8)
        mask = np.empty((self.G, self.C), np.uint8)
        reward = np.empty(self.G, np.float32)
        done = np.empty(self.G, np.uint8)
        term = np.zeros((self.G, self.N, self.N), np.int8) if want_term else None
        aout = np.empty(self.G, np.int32)
        a = None if actions is None else np.ascontiguousarray(actions, np.int32)
        u = None if opp_u is None else np.ascontiguousarray(opp_u, np.float64)
        lib().emu_step(self._h, _p(a), _p(u), _p(obs), _p(mask), _p(reward), _p(done), _p(term), _p(aout))
        out = dict(obs=obs, mask=mask, reward=reward, done=done, actions=aout)
        if want_term:
            out["term_obs"] = term
        return out

    def half_step(self, side, actions, want_term=False):
        reward = np.empty(self.G, np.float32)
        done = np.empty(self.G, np.uint8)
        term = np.zeros((self.G, self.N, self.N), np.int8) if want_term else None
        a = None if actions is None else np.ascontiguousarray(actions, np.int32)
        lib().emu_half_step(self._h, side, _p(a), _p(reward), _p(done), _p(term))
        out = dict(reward=reward, done=done, to_move=self.to_move.copy(), opp_index=self.opp_index.copy())
        if want_term:
            out["term_obs"] = term
        return out

    def rollout(self, T, want_term=False):
        G, N, C = self.G, self.N, self.C
        out = dict(obs=np.empty((T, G, N, N), np.int8), mask=np.empty((T, G, C), np.uint8), reward=np.empty((T, G), np.float32),
                   done=np.empty((T, G), np.uint8), term_obs=np.zeros((T, G, N, N), np.int8), actions=np.empty((T, G), np.int32))
        lib().emu_rollout(self._h, T, _p(out["obs"]), _p(out["mask"]), _p(out["reward"]), _p(out["done"]),
                          _p(out["term_obs"]) if want_term else None, _p(out["actions"]))
        return out

    def enable_info(self):
        self.info_opp = np.full(self.G, -1, np.int32)
        self.info_winner = np.full(self.G, -1, np.int8)
        lib().emu_set_info(self._h, _p(self.info_opp), _p(self.info_winner))

    def info(self):
        return self.info_opp.copy(), self.info_winner.copy()

    def opp_state(self):
        return self.to_move.copy(), self.opp_index.copy()

    def view1(self):
        return self.encode(1)

    def ply(self, actions):
        ret = np.empty(self.G, np.int8)
        a = np.ascontiguousarray(actions, np.int32)
        lib().emu_ply(self._h, _p(a), _p(ret))
        return ret

    def encode(self, view=0):
        obs = np.empty((self.G, self.N, self.N), np.int8)
        mask = np.empty((self.G, self.C), np.uint8)
        lib().emu_encode(self._h, view, _p(obs), _p(mask))
        return obs, mask

    def sample_actions(self, u, view=0):
        out = np.empty(self.G, np.int32)
        uu = np.ascontiguousarray(u, np.float64)
        lib().emu_sample_actions(self._h, view, _p(uu), _p(out))
        return out

    def import_boards(self, board_true, to_move=None, import_mask=None):
        b = np.ascontiguousarray(board_true, np.int8)
        tm = None if to_move is None else np.ascontiguousarray(to_move, np.int8)
        im = None if import_mask is None else np.ascontiguousarray(import_mask, np.uint8)
        lib().emu_import_boards(self._h, _p(b), _p(tm), _p(im))

    def import_labels(self, board_true, regions, to_move=None, import_mask=None):
        b = np.ascontiguousarray(board_true, np.int8)
        r = np.ascontiguousarray(regions, np.uint8)
        tm = None if to_move is None else np.ascontiguousarray(to_move, np.int8)
        im = None if import_mask is None else np.ascontiguousarray(import_mask, np.uint8)
        lib().emu_import_labels(self._h, _p(b), _p(r), _p(tm), _p(im))

    def opponent_catch_up(self):
        lib().emu_half_step(self._h, 1, None, None, None, None)

    def export(self):
        N, G = self.N, self.G
        out = dict(board=np.empty((G, N, N), np.float64), regions=np.empty((G, 2, N + 2, N + 2), np.float64),
                   region_counter=np.empty((G, 2), np.float64), cur=np.empty(G, np.int8), done=np.empty(G, np.uint8),
                   winner=np.empty(G, np.int8), agent=np.empty(G, np.int8), draws=np.empty(G, np.uint32))
        lib().emu_export_state(self._h, *[_p(out[k]) for k in
                                          ("board", "regions", "region_counter", "cur", "done", "winner", "agent", "draws")])
        return out

    def stats(self):
        out = np.zeros(8, np.int64)
        lib().emu_stats(self._h, _p(out))
        return out


def copy_games(dst, src, src_index=None, dst_index=None, count=None):
    """hexb_copy_games between two EmuBatch objects (dst raw, same N and variant)."""
    si = None if src_index is None else np.ascontiguousarray(src_index, np.int64)
    di = None if dst_index is None else np.ascontiguousarray(dst_index, np.int64)
    if count is None:
        count = len(si) if si is not None else (len(di) if di is not None else min(dst.G, src.G))
    lib().emu_copy_games(dst._h, src._h, _p(si), _p(di), int(count))


def _policy(policy):
    if policy not in POLICIES:
        raise ValueError("policy must be 0 (random) or 1 (bridge)")
    return int(policy)


def playouts(batch, num_playouts, first_playout=0, game_mask=None, policy=0):
    """hexb_playouts_policy on an EmuBatch: wins i32[G]."""
    policy = _policy(policy)
    wins = np.empty(batch.G, np.int32)
    gm = None if game_mask is None else np.ascontiguousarray(game_mask, np.uint8)
    lib().emu_playouts(batch._h, int(num_playouts), int(first_playout), policy, _p(gm), _p(wins))
    return wins


class EmuMCTS(object):
    """hexb_mcts_* on an EmuBatch, with the method surface of hex_gym_env_b200.MCTS (numpy in and out)."""

    def __init__(self, batch, max_nodes, c_puct=1.25, fpu=0.0):
        self.batch, self.max_nodes, self.c_puct, self.fpu = batch, int(max_nodes), float(c_puct), float(fpu)
        self.tree = np.zeros(int(lib().emu_mcts_tree_bytes(batch.N, batch.G, self.max_nodes)), np.uint8)

    def _call(self, op, first_playout=0, root_mask=None, sims=0, playouts=0, policy=0, **out):
        ptrs = [_p(out.get(k)) for k in ("leaf_obs", "leaf_mask", "pending", "priors", "values", "visits", "q", "value", "nodes_used")]
        lib().emu_mcts(self.batch._h, op, _p(self.tree), self.tree.size, self.max_nodes, self.c_puct, self.fpu, int(first_playout),
                       _p(root_mask), int(sims), int(playouts), policy, *ptrs)

    def reset(self, root_mask=None, first_playout=0):
        rm = None if root_mask is None else np.ascontiguousarray(root_mask, np.uint8)
        self._call(MCTS_INIT, first_playout, rm)

    def search(self, num_simulations, playouts_per_leaf, policy=0):
        self._call(MCTS_SEARCH, sims=num_simulations, playouts=playouts_per_leaf, policy=_policy(policy))

    def select(self):
        G, N, C = self.batch.G, self.batch.N, self.batch.C
        obs, mask, pending = np.zeros((G, N, N), np.int8), np.zeros((G, C), np.uint8), np.zeros(G, np.uint8)
        self._call(MCTS_SELECT, leaf_obs=obs, leaf_mask=mask, pending=pending)
        return obs, mask, pending

    def expand(self, priors, values):
        self._call(MCTS_EXPAND, priors=np.ascontiguousarray(priors, np.float32), values=np.ascontiguousarray(values, np.float32))

    def root(self):
        G, C = self.batch.G, self.batch.C
        out = dict(visits=np.zeros((G, C), np.int32), q=np.zeros((G, C), np.float32), value=np.zeros(G, np.float32),
                   nodes_used=np.zeros(G, np.int32))
        self._call(MCTS_ROOT, **out)
        return out["visits"], out["q"], out["value"], out["nodes_used"]

    def advance(self, root_mask=None, first_playout=0):
        rm = None if root_mask is None else np.ascontiguousarray(root_mask, np.uint8)
        self._call(MCTS_ADVANCE, first_playout, rm)
