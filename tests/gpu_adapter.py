"""Adapter giving hex_gym_env_b200.HexBatch (CUDA, through the C ABI) the numpy method surface of oracle.hexref.RefBatch
so that tests/parity.py can drive it. Used only by the -m gpu tests."""
import numpy as np
import torch

from hex_gym_env_b200 import HexBatch
from oracle import hexref


class GpuBatch(object):
    def __init__(self, variant, N, G, launch_form=0, obs_f32=False, **kw):
        self.b = HexBatch(N, G, variant=variant, device=0, obs_dtype=torch.float32 if obs_f32 else torch.int8, **kw)
        if launch_form:
            self.b.set_launch_form(launch_form)   # 1 / 4 warps per chunk instead of the depth-based choice
        self.N, self.G = N, G

    @staticmethod
    def _np(t):
        a = t.cpu().numpy()
        if a.dtype == np.float32 and a.ndim >= 3:   # float32 observations (obs_dtype f32) hold the same small integers
            b = a.astype(np.int8)
            assert np.array_equal(b.astype(np.float32), a), "float32 observation with a non-integer value"
            return b
        return a

    def reset(self, reset_mask=None, open_u=None):
        obs, mask = self.b.reset(reset_mask, open_u)
        return self._np(obs), self._np(mask)

    def step(self, actions=None, opp_u=None, want_term=False):
        if want_term:
            self.b._buf("term_obs", (self.G, self.N, self.N), self.b.obs_dtype).zero_()
        o = self.b.step(actions, opp_u, want_term=want_term, want_actions=True)
        return {k: self._np(v) for k, v in o.items()}

    def half_step(self, side, actions, want_term=False):
        if want_term:
            self.b._buf("term_obs", (self.G, self.N, self.N), self.b.obs_dtype).zero_()
        o = self.b.half_step(side, actions, want_term=want_term)
        out = {k: self._np(v) for k, v in o.items()}
        out["to_move"], out["opp_index"] = self.opp_state()
        return out

    def rollout(self, T, want_term=False):
        G, N = self.G, self.N
        term = torch.zeros((T, G, N, N), dtype=self.b.obs_dtype, device="cuda") if want_term else None
        acts = torch.empty((T, G), dtype=torch.int32, device="cuda")
        o = self.b.rollout(T, term_obs=term, actions_out=acts)
        return {k: self._np(v) for k, v in o.items()}

    def enable_info(self):
        self.b.enable_info()

    def info(self):
        return self._np(self.b.last_move_opponent), self._np(self.b.winner)

    def opp_state(self):
        return self._np(self.b.to_move), self._np(self.b.opp_index)

    def set_eval(self, eval_state):
        self.b.set_eval(eval_state)

    def set_opponent_eps(self, eps):
        self.b.set_opponent_eps(eps)

    def view1(self):
        return self.encode(1)

    def ply(self, actions):
        return self._np(self.b.ply(actions))

    def encode(self, view=0):
        obs, mask = self.b.encode(view)
        return self._np(obs), self._np(mask)

    def sample_actions(self, u, view=0):
        return self._np(self.b.sample_actions(u, view))

    def import_boards(self, board_true, to_move=None, import_mask=None):
        self.b.import_boards(board_true, to_move, import_mask)

    def import_labels(self, board_true, regions, to_move=None, import_mask=None):
        self.b.import_labels(board_true, regions, to_move, import_mask)

    def opponent_catch_up(self):
        self.b.opponent_catch_up()

    def export(self):
        e = {k: self._np(v) for k, v in self.b.export_state().items()}
        e["draws"] = e["draws"].astype(np.uint32)
        return e

    def stats(self):
        return self._np(self.b.stats())


def make(kind, N, G, seed=0, game_offset=0, agent_mode=0, opponent_first=False, auto_reset=True, eval_state=False,
         manual_opponent=False, pool_size=0, launch_form=0, obs_f32=False):
    if kind == hexref.KIND_GAME_A:
        return GpuBatch(0, N, G, raw=True)
    variant = 0 if kind == hexref.KIND_ENV_A else 1
    return GpuBatch(variant, N, G, seed=seed, game_offset=game_offset, agent_mode=agent_mode, opponent_first=opponent_first,
                    auto_reset=auto_reset, eval_state=eval_state, manual_opponent=manual_opponent, pool_size=pool_size,
                    launch_form=launch_form, obs_f32=obs_f32)


def make_with(**fixed):
    """`make` with some keyword arguments pinned (launch_form=..., obs_f32=...): the drivers in tests/parity.py pass the rest."""
    def mk(kind, N, G, **kw):
        kw.update(fixed)
        if kind == hexref.KIND_GAME_A:
            return make(kind, N, G)
        return make(kind, N, G, **kw)
    return mk
