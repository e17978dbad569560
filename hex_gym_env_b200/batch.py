"""HexBatch - G independent Hex games living on one B200, advanced in lockstep by the kernels of libhexb.so.

This is the thin host object over the C ABI of include/hexb.h. torch is used for device memory, streams and
(in multi_gpu.py) torch.distributed only; every operation on game state is a call through the C ABI into the
hand-written sm_100a kernels (hex_gym_env_b200/csrc). There is no CPU path: constructing a HexBatch without the
CUDA library or without a GPU raises.

What each method replaces in the reference (MBPrdctns/hex_gym_env, paths relative to its root):
  reset()            HexEnv.reset (minihex/HexGame.py:206-242, minihex/HexSingleGame.py:208-231), SelfPlayEnv.reset
                     (minihex/SelfplayWrapper.py:69-89) for all games or a masked subset
  step()             SelfPlayEnv.step (SelfplayWrapper.py:174-199) / variant-A HexEnv.step (HexGame.py:244-295) incl. the
                     random opponent, reward/done, DummyVecEnv-style auto-reset, observation and legal-action mask
  ply()              HexGame.make_move / fast_move (HexGame.py:85-111, HexSingleGame.py:88-122)
  encode()           get_action_mask (HexGame.py:203-204) / legal_actions (HexSingleGame.py:205-206) + the live board
  sample_actions()   BaseRandomPolicy.choose_action (SelfplayWrapper.py:17-22) / random_policy (minihex/__init__.py:8-12)
  export_state()     attribute reads .board / .regions / .region_counter / .current_player_num / .done / .winner
  import_boards()    HexGame.__init__ with a preset board (HexGame.py:53-61, HexSingleGame.py:57-65)
  copy_games()       copy.deepcopy(env.simulator) into a raw batch (tree search: branching a position)
  playouts()         random playouts to the end from the current position (tree search: Monte-Carlo value estimates)
"""
import ctypes
import os

import torch

from . import _native
from ._native import HexbConfig, check

VARIANT_A = 0  # minihex/HexGame.py
VARIANT_B = 1  # minihex/HexSingleGame.py + minihex/SelfplayWrapper.py
AGENT_BLACK, AGENT_WHITE, AGENT_RANDOM = 0, 1, 2

STAT_NAMES = ("episodes", "black_wins", "white_wins", "agent_wins", "episode_plies", "invalid_ends", "env_steps", "plies")
COMPRESSIBLE_MIN_BYTES = 8 << 20   # smaller buffers stay with torch's allocator even when the object uses compressible memory


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class HexBatch(object):
    def __init__(self, board_size, num_games, variant=VARIANT_B, device=None, seed=0, game_offset=0,
                 agent_mode=AGENT_BLACK, opponent_first=False, auto_reset=True, eval_state=False, raw=False,
                 manual_opponent=False, pool_size=0, obs_dtype=torch.int8, compressible=None):
        self._h = None
        self._lib = _native.lib()  # raises if libhexb.so cannot be built / loaded
        if not torch.cuda.is_available():
            raise RuntimeError("hex_gym_env_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.N, self.G, self.C = int(board_size), int(num_games), int(board_size) * int(board_size)
        self.variant, self.raw, self.auto_reset = int(variant), bool(raw), bool(auto_reset)
        if obs_dtype not in (torch.int8, torch.float32):
            raise ValueError("obs_dtype must be torch.int8 or torch.float32")
        self.obs_dtype = obs_dtype   # element type of every obs / term_obs tensor (hexb_config.obs_dtype)
        self.cfg = HexbConfig(board_size=self.N, variant=self.variant, num_games=self.G, game_offset=int(game_offset),
                              seed=int(seed) & 0xFFFFFFFFFFFFFFFF, agent_mode=int(agent_mode), opponent_first=int(bool(opponent_first)),
                              auto_reset=int(bool(auto_reset)), eval_state=int(bool(eval_state)), raw=int(bool(raw)),
                              device=self.device.index, manual_opponent=int(bool(manual_opponent)), pool_size=int(pool_size),
                              obs_dtype=1 if obs_dtype == torch.float32 else 0)
        self.manual_opponent = bool(manual_opponent)
        nbytes = self._lib.hexb_state_bytes(ctypes.byref(self.cfg))
        if nbytes == 0:
            raise ValueError("unsupported configuration: board_size=%r num_games=%r variant=%r agent_mode=%r"
                             % (board_size, num_games, variant, agent_mode))
        self.state_bytes = int(nbytes)
        # Compressible device memory (hexb_mem_alloc) for the packed state and the object's own large output tensors: the L2's inline
        # compression then shrinks their HBM traffic (label bytes, -1/0/+1 observations and 0/1 masks compress well): 1 Mi games of
        # 19x19 244 -> 187-209 us per step, 11x11 88.1 -> 86.5. Only deep launches are bound by HBM, so the default is by size
        # (state of at least 64 MiB); compressible=True / False or HEXB_COMPRESSIBLE=1 / 0 force it. memory_kind says what was granted.
        if compressible is None:
            env_c = os.environ.get("HEXB_COMPRESSIBLE")
            compressible = (env_c != "0") if env_c is not None else self.state_bytes >= (64 << 20)
        self.compressible = bool(compressible)
        self.memory_kind = "ordinary (torch allocator)"
        with torch.cuda.device(self.device):
            self._state = self._alloc(self.state_bytes + 256)
            off = (-self._state.data_ptr()) % 256
            self._state_ptr = self._state.data_ptr() + off
            h = ctypes.c_void_p()
            check(self._lib.hexb_create(ctypes.byref(self.cfg), ctypes.c_void_p(self._state_ptr), self.state_bytes,
                                        self._stream(), ctypes.byref(h)))
        self._h = h
        self.opp_index = self.to_move = self.eval_episode = None
        if manual_opponent:  # per-game opponent bookkeeping, written by every reset / half step
            self.opp_index = torch.full((self.G,), -1, dtype=torch.int32, device=self.device)
            self.to_move = torch.full((self.G,), 2, dtype=torch.uint8, device=self.device)
            check(self._lib.hexb_set_opponent_buffers(self._h, _ptr(self.opp_index), _ptr(self.to_move)))
            if eval_state:   # the evaluation cycle through the pool needs its per-game episode counter
                self.set_eval(True)
        self._out = {}
        self._ws = None
        self._pinned = None
        self._packed = None

    # ------------------------------------------------------------------ plumbing
    @property
    def handle(self):
        """The hexb_env* as an int: the first argument of the torch.ops.hexb.* operators (torch_ops.py)."""
        return int(self._h.value)

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.hexb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _alloc(self, nbytes):
        """uint8[nbytes] on the device: compressible memory from the library for large buffers when enabled, else torch's allocator."""
        if self.compressible and nbytes >= COMPRESSIBLE_MIN_BYTES:
            try:
                buf = _native.DeviceBuffer(nbytes, self.device.index, True)
                self.memory_kind = "compressible (cuMemCreate, CU_MEM_ALLOCATION_COMP_GENERIC)" if buf.compressed else \
                    "ordinary (hexb_mem_alloc: the driver did not grant compression)"
                return torch.as_tensor(buf, device=self.device)
            except Exception as exc:   # no VMM / out of address space: ordinary memory does the same job
                self.compressible = False
                self.memory_kind = "ordinary (torch allocator; hexb_mem_alloc failed: %s)" % exc
        return torch.empty(nbytes, dtype=torch.uint8, device=self.device)

    def _buf(self, name, shape, dtype):
        t = self._out.get(name)
        if t is None:
            n = 1
            for d in shape:
                n *= int(d)
            nbytes = n * torch.empty((), dtype=dtype).element_size()
            if self.compressible and nbytes >= COMPRESSIBLE_MIN_BYTES:
                t = self._alloc(nbytes)[:nbytes].view(dtype).reshape(shape)
            else:
                t = torch.empty(shape, dtype=dtype, device=self.device)
            self._out[name] = t
        return t

    def _chk(self, t, shape, dtype, name):
        if t is None:
            return None
        if not (t.is_cuda and t.device == self.device and t.dtype == dtype and t.is_contiguous() and tuple(t.shape) == tuple(shape)):
            raise ValueError("%s must be a contiguous %s tensor of shape %s on %s" % (name, dtype, tuple(shape), self.device))
        return t

    def _in(self, x, shape, dtype, name):
        if x is None:
            return None
        t = torch.as_tensor(x)
        if t.dtype != dtype or not t.is_cuda or t.device != self.device:
            t = t.to(device=self.device, dtype=dtype)
        t = t.contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError("%s must have shape %s, got %s" % (name, tuple(shape), tuple(t.shape)))
        return t

    # ------------------------------------------------------------------ the hot path
    def reset(self, reset_mask=None, open_u=None, obs=None, mask=None):
        """Reset all games (or those with reset_mask != 0). Returns (obs i8[G,N,N], mask u8[G,C]) device tensors."""
        G, N, C = self.G, self.N, self.C
        rm = self._in(reset_mask, (G,), torch.uint8, "reset_mask")
        ou = self._in(open_u, (G,), torch.float64, "open_u")
        obs = self._chk(obs, (G, N, N), self.obs_dtype, "obs") if obs is not None else self._buf("obs", (G, N, N), self.obs_dtype)
        mask = self._chk(mask, (G, C), torch.uint8, "mask") if mask is not None else self._buf("mask", (G, C), torch.uint8)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_reset(self._h, _ptr(rm), _ptr(ou), _ptr(obs), _ptr(mask), self._stream()))
        return obs, mask

    def step(self, actions=None, opp_u=None, obs=None, mask=None, reward=None, done=None, term_obs=None, actions_out=None,
             want_term=False, want_actions=False, outputs=True):
        """One env step for every game. actions=None: the agent is the random policy as well (fused sampling).

        Returns a dict of device tensors (obs, mask, reward, done [, term_obs, actions]). The default output tensors
        are owned by this object and overwritten by the next call (like the reference, whose observation is the live
        board array); pass your own tensors (e.g. rollout-buffer slices) to keep them. outputs=False steps without
        writing any observation (pure simulation)."""
        G, N, C = self.G, self.N, self.C
        a = self._in(actions, (G,), torch.int32, "actions")
        u = self._in(opp_u, (G, 2), torch.float64, "opp_u")
        if outputs:
            obs = self._chk(obs, (G, N, N), self.obs_dtype, "obs") if obs is not None else self._buf("obs", (G, N, N), self.obs_dtype)
            mask = self._chk(mask, (G, C), torch.uint8, "mask") if mask is not None else self._buf("mask", (G, C), torch.uint8)
            reward = self._chk(reward, (G,), torch.float32, "reward") if reward is not None else self._buf("reward", (G,), torch.float32)
            done = self._chk(done, (G,), torch.uint8, "done") if done is not None else self._buf("done", (G,), torch.uint8)
        if term_obs is not None:
            term_obs = self._chk(term_obs, (G, N, N), self.obs_dtype, "term_obs")
        elif want_term:
            term_obs = self._buf("term_obs", (G, N, N), self.obs_dtype)
        if actions_out is not None:
            actions_out = self._chk(actions_out, (G,), torch.int32, "actions_out")
        elif want_actions:
            actions_out = self._buf("actions", (G,), torch.int32)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_step(self._h, _ptr(a), _ptr(u), _ptr(obs), _ptr(mask), _ptr(reward), _ptr(done), _ptr(term_obs),
                                      _ptr(actions_out), self._stream()))
        out = dict(obs=obs, mask=mask, reward=reward, done=done)
        if term_obs is not None:
            out["term_obs"] = term_obs
        if actions_out is not None:
            out["actions"] = actions_out
        return out

    def rollout(self, num_steps, obs=None, mask=None, reward=None, done=None, term_obs=None, actions_out=None, outputs=True):
        """num_steps env steps in ONE launch with the fused random agent (= step(actions=None) called num_steps times, bit for
        bit), the state staying on chip in between. Outputs have a leading step dimension, like a rollout buffer:
        obs i8[T,G,N,N], mask u8[T,G,C], reward f32[T,G], done u8[T,G] (+ term_obs, actions_out when given)."""
        T, G, N, C = int(num_steps), self.G, self.N, self.C
        if outputs:
            obs = self._chk(obs, (T, G, N, N), self.obs_dtype, "obs") if obs is not None else self._buf("r_obs%d" % T, (T, G, N, N), self.obs_dtype)
            mask = self._chk(mask, (T, G, C), torch.uint8, "mask") if mask is not None else self._buf("r_mask%d" % T, (T, G, C), torch.uint8)
            reward = self._chk(reward, (T, G), torch.float32, "reward") if reward is not None else self._buf("r_rew%d" % T, (T, G), torch.float32)
            done = self._chk(done, (T, G), torch.uint8, "done") if done is not None else self._buf("r_done%d" % T, (T, G), torch.uint8)
        term_obs = self._chk(term_obs, (T, G, N, N), self.obs_dtype, "term_obs")
        actions_out = self._chk(actions_out, (T, G), torch.int32, "actions_out")
        with torch.cuda.device(self.device):
            check(self._lib.hexb_rollout(self._h, T, _ptr(obs), _ptr(mask), _ptr(reward), _ptr(done), _ptr(term_obs), _ptr(actions_out),
                                         self._stream()))
        out = dict(obs=obs, mask=mask, reward=reward, done=done)
        if term_obs is not None:
            out["term_obs"] = term_obs
        if actions_out is not None:
            out["actions"] = actions_out
        return out

    def capture_steps(self, num_steps, **step_kwargs):
        """Capture `num_steps` calls of step(**step_kwargs) into a CUDA graph and return it (torch.cuda.CUDAGraph; .replay()
        runs the steps on the current stream). For launch-bound batches: a 65,536-game 7x7 step is 8 us on the device but
        12 us to issue from Python. The graph reads and writes the tensors passed in step_kwargs (or this object's default
        output tensors): refill an `actions` tensor in place between replays. One eager step runs first (outside the graph)."""
        dev = self.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            self.step(**step_kwargs)          # allocates the default output tensors and loads the kernel before the capture
            side.synchronize()
            with torch.cuda.graph(graph, stream=side):
                for _ in range(int(num_steps)):
                    out = self.step(**step_kwargs)
        torch.cuda.current_stream(dev).wait_stream(side)
        graph.outputs = out
        return graph

    def enable_info(self):
        """Also record, at every step(), the fields of the reference's info dict (HexGame.py:281-286) as device tensors:
        self.last_move_opponent i32[G] and self.winner i8[G]; info["last_move_player"] is step(want_actions=True)["actions"]."""
        self.last_move_opponent = torch.full((self.G,), -1, dtype=torch.int32, device=self.device)
        self.winner = torch.full((self.G,), -1, dtype=torch.int8, device=self.device)
        check(self._lib.hexb_set_info_buffers(self._h, _ptr(self.last_move_opponent), _ptr(self.winner)))
        return self.last_move_opponent, self.winner

    def pinned_io(self):
        """Pinned host buffers for step_host: dict(actions i32[G], obs i8[G,N,N], mask u8[G,C], reward f32[G], done u8[G])."""
        if self._pinned is None:
            G, N, C = self.G, self.N, self.C
            self._pinned = dict(actions=torch.empty(G, dtype=torch.int32).pin_memory(),
                                obs=torch.empty((G, N, N), dtype=self.obs_dtype).pin_memory(),
                                mask=torch.empty((G, C), dtype=torch.uint8).pin_memory(),
                                reward=torch.empty(G, dtype=torch.float32).pin_memory(),
                                done=torch.empty(G, dtype=torch.uint8).pin_memory())
        return self._pinned

    def set_launch_form(self, warps_per_chunk=0):
        """0: the kernel form is chosen by launch depth; 1 / 4: that many warps per 32-game chunk (tests). Other values raise HexbError."""
        check(self._lib.hexb_set_launch_form(self._h, int(warps_per_chunk)))

    def set_host_transport(self, dma_fraction=-1.0):
        """How step_host moves obs + mask: share of the games copied as plain bytes by DMA, the rest as 2 bits per cell expanded
        by host threads. Negative = adaptive (default), 1.0 = plain DMA only, 0.0 = everything packed."""
        check(self._lib.hexb_set_host_transport(self._h, float(dma_fraction)))

    def host_transport(self):
        f = ctypes.c_double()
        check(self._lib.hexb_get_host_transport(self._h, ctypes.byref(f)))
        return f.value

    def _host_actions(self, actions_host, io):
        """Pointer to the step's host actions: a contiguous int32 CPU tensor (e.g. a row of a pinned trajectory) is used as it
        is; anything else is staged through io["actions"]."""
        if actions_host is None:
            return None
        if isinstance(actions_host, torch.Tensor) and actions_host.dtype == torch.int32 and not actions_host.is_cuda \
                and actions_host.is_contiguous() and actions_host.numel() == self.G:
            return _ptr(actions_host)
        io["actions"].copy_(torch.as_tensor(actions_host, dtype=torch.int32))
        return _ptr(io["actions"])

    def _host_ws(self):
        if self._ws is None:
            n = self._lib.hexb_host_workspace_bytes(ctypes.byref(self.cfg))
            self._ws = torch.empty(int(n) + 256, dtype=torch.uint8, device=self.device)
        return ctypes.c_void_p(self._ws.data_ptr() + ((-self._ws.data_ptr()) % 256))

    def step_host_begin(self, actions_host=None, io=None, want_obs=True, want_mask=True):
        """step_host split in two: enqueue H2D + step + D2H and return at once (a host-side policy can work meanwhile);
        step_host_end() waits until `io` holds the results. One step may be pending."""
        io = io or self.pinned_io()
        ap = self._host_actions(actions_host, io)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_step_host_begin(self._h, self._host_ws(), ap,
                                                 _ptr(io["obs"]) if want_obs else None, _ptr(io["mask"]) if want_mask else None,
                                                 _ptr(io["reward"]), _ptr(io["done"]), self._stream()))
        return io

    def step_host_end(self):
        with torch.cuda.device(self.device):
            check(self._lib.hexb_step_host_end(self._h))

    def step_host_packed(self, actions_host=None, io=None):
        """step_host with the observations crossing PCIe as 2 bits per cell; host threads expand them into io["obs"] / io["mask"]
        (bit-identical to step_host; int8 observations only)."""
        io = io or self.pinned_io()
        if self._packed is None:
            n = int(self._lib.hexb_host_packed_bytes(ctypes.byref(self.cfg)))
            self._packed = torch.empty(n + 64, dtype=torch.uint8).pin_memory()
        ph = self._packed.data_ptr() + ((-self._packed.data_ptr()) % 64)
        ap = self._host_actions(actions_host, io)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_step_host_packed(self._h, self._host_ws(), ctypes.c_void_p(ph), ap, _ptr(io["obs"]),
                                                  _ptr(io["mask"]), _ptr(io["reward"]), _ptr(io["done"]), self._stream()))
        return io

    def step_host(self, actions_host=None, io=None, want_obs=True, want_mask=True):
        """The step as a host-side user of the reference API makes it: HOST actions in, HOST obs/mask/reward/done out
        (one call, copies inside, returns when the results are in host memory). `io` = pinned_io() or compatible CPU
        tensors. actions_host=None: fused agent sampling on the device (no H2D)."""
        io = io or self.pinned_io()
        ap = self._host_actions(actions_host, io)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_step_host(self._h, self._host_ws(), ap,
                                           _ptr(io["obs"]) if want_obs else None, _ptr(io["mask"]) if want_mask else None,
                                           _ptr(io["reward"]), _ptr(io["done"]), self._stream()))
        return io

    # ------------------------------------------------------------------ learned opponent (manual_opponent=True)
    def half_step(self, side, actions, reward=None, done=None, term_obs=None, want_term=False):
        """One ply of `side` (0 agent, 1 opponent) in every game whose turn it is; actions i32[G] in the mover's own view.
        Returns dict(reward, done [, term_obs]); self.to_move / self.opp_index are updated in place."""
        G, N = self.G, self.N
        a = self._in(actions, (G,), torch.int32, "actions")   # None (side 1 only): the built-in random opponent moves
        reward = self._chk(reward, (G,), torch.float32, "reward") if reward is not None else self._buf("h_reward%d" % side, (G,), torch.float32)
        done = self._chk(done, (G,), torch.uint8, "done") if done is not None else self._buf("h_done%d" % side, (G,), torch.uint8)
        if term_obs is not None:
            term_obs = self._chk(term_obs, (G, N, N), self.obs_dtype, "term_obs")
        elif want_term:
            term_obs = self._buf("term_obs", (G, N, N), self.obs_dtype)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_half_step(self._h, int(side), _ptr(a), _ptr(reward), _ptr(done), _ptr(term_obs), self._stream()))
        out = dict(reward=reward, done=done)
        if term_obs is not None:
            out["term_obs"] = term_obs
        return out

    def set_eval(self, eval_state):
        """SelfPlayEnv.set_eval (SelfplayWrapper.py:117-120) for every game of the batch, at run time: while it is on, a restart
        draws nothing for the opponent choice and - on a manual_opponent batch - episode k of a game since this call meets pool
        entry k (self.opp_index = k while k <= pool_size - 1, then it stays; setup_opponents :92-96). Episodes under way go on."""
        if self.variant != VARIANT_B or self.raw:
            raise ValueError("set_eval belongs to SelfPlayEnv (variant B env handles)")
        if self.opp_index is not None and self.eval_episode is None:
            self.eval_episode = torch.zeros(self.G, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_set_eval(self._h, int(bool(eval_state)), _ptr(self.eval_episode), self._stream()))
        self.cfg.eval_state = int(bool(eval_state))

    opponent_eps = None   # what set_opponent_eps last set (None: the caller's action always)

    def set_opponent_eps(self, eps):
        """Variant-A HexEnv(opponent_policy="opponent_predict", eps=...) (HexGame.py:354-359) on a manual_opponent batch: every
        opponent half step first draws rv from the game's stream and lets random_policy move when rv < eps, else plays the
        caller's action (the model's prediction on encode(1)). eps=None or negative: the caller's action always."""
        check(self._lib.hexb_set_opponent_eps(self._h, -1.0 if eps is None else float(eps)))
        self.opponent_eps = None if eps is None or eps < 0 else float(eps)

    @property
    def eval_state(self):
        return bool(self.cfg.eval_state)

    def opponent_opening(self, opponent_fn):
        """After reset(): let the caller's opponent open the games in which it moves first (agent is WHITE)."""
        o1, m1 = self._buf("opp_obs", (self.G, self.N, self.N), self.obs_dtype), self._buf("opp_mask", (self.G, self.C), torch.uint8)
        self.encode(1, obs=o1, mask=m1)
        self.half_step(1, opponent_fn(o1, m1, self.to_move, self.opp_index))

    def step_with_opponent(self, actions, opponent_fn, want_term=False, obs=None, mask=None):
        """One env step against a learned opponent, all on the device: agent ply, then up to two opponent plies (the reply,
        and the opening move of a game that restarted with the opponent to move). `opponent_fn(obs i8[G,N,N], mask u8[G,C],
        to_move u8[G], opp_index i32[G]) -> actions i32[G]` sees the side-to-move view (what OpponentPolicy.choose_action gets,
        SelfplayWrapper.py:161) and must answer for the games with to_move == 1; its other entries are ignored."""
        G, N, C = self.G, self.N, self.C
        term = self._buf("sw_term", (G, N, N), self.obs_dtype) if want_term else None
        h = self.half_step(0, actions, term_obs=term)
        reward, done = h["reward"].clone(), h["done"].clone()
        o1, m1 = self._buf("opp_obs", (G, N, N), self.obs_dtype), self._buf("opp_mask", (G, C), torch.uint8)
        for _ in range(2):
            self.encode(1, obs=o1, mask=m1)
            h = self.half_step(1, opponent_fn(o1, m1, self.to_move, self.opp_index), term_obs=term)
            reward += h["reward"]
            done |= h["done"]
        obs, mask = self.encode(0, obs=obs, mask=mask)
        out = dict(obs=obs, mask=mask, reward=reward, done=done)
        if want_term:
            out["term_obs"] = term
        return out

    # ------------------------------------------------------------------ the pieces on their own
    def ply(self, actions, ret=None):
        a = self._in(actions, (self.G,), torch.int32, "actions")
        ret = self._chk(ret, (self.G,), torch.int8, "ret") if ret is not None else self._buf("ret", (self.G,), torch.int8)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_ply(self._h, _ptr(a), _ptr(ret), self._stream()))
        return ret

    def encode(self, view=0, obs=None, mask=None):
        G, N, C = self.G, self.N, self.C
        obs = self._chk(obs, (G, N, N), self.obs_dtype, "obs") if obs is not None else self._buf("obs", (G, N, N), self.obs_dtype)
        mask = self._chk(mask, (G, C), torch.uint8, "mask") if mask is not None else self._buf("mask", (G, C), torch.uint8)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_encode(self._h, int(view), _ptr(obs), _ptr(mask), self._stream()))
        return obs, mask

    def sample_actions(self, u, view=0, out=None):
        uu = self._in(u, (self.G,), torch.float64, "u")
        out = self._chk(out, (self.G,), torch.int32, "out") if out is not None else self._buf("sampled", (self.G,), torch.int32)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_sample_actions(self._h, int(view), _ptr(uu), _ptr(out), self._stream()))
        return out

    def export_state(self):
        """Reference-layout dump (float64 like the reference's numpy arrays). New tensors every call."""
        G, N = self.G, self.N
        dev = self.device
        out = dict(board=torch.empty((G, N, N), dtype=torch.float64, device=dev),
                   regions=torch.empty((G, 2, N + 2, N + 2), dtype=torch.float64, device=dev),
                   region_counter=torch.empty((G, 2), dtype=torch.float64, device=dev),
                   cur=torch.empty(G, dtype=torch.int8, device=dev), done=torch.empty(G, dtype=torch.uint8, device=dev),
                   winner=torch.empty(G, dtype=torch.int8, device=dev), agent=torch.empty(G, dtype=torch.int8, device=dev),
                   draws=torch.empty(G, dtype=torch.int32, device=dev))
        with torch.cuda.device(self.device):
            check(self._lib.hexb_export_state(self._h, *[_ptr(out[k]) for k in ("board", "regions", "region_counter", "cur", "done",
                                                                                 "winner", "agent", "draws")], self._stream()))
        return out

    def export_state_host(self, ply_actions=None):
        """export_state() for host readers (the single-game drop-in classes): ONE kernel into one packed device buffer, ONE
        device->host copy into pinned memory, numpy views on it. The arrays are overwritten by the next call.
        ply_actions (host ints, raw handles): first play these moves (hexb_ply) in the same round trip; the dict then also
        holds "ret" (HexGame.make_move's return codes)."""
        G, N = self.G, self.N
        spec = (("board", (G, N, N), torch.float64), ("regions", (G, 2, N + 2, N + 2), torch.float64),
                ("region_counter", (G, 2), torch.float64), ("draws", (G,), torch.int32), ("cur", (G,), torch.int8),
                ("done", (G,), torch.uint8), ("winner", (G,), torch.int8), ("agent", (G,), torch.int8), ("ret", (G,), torch.int8))
        if getattr(self, "_xdev", None) is None:
            off, views = 0, []
            for name, shape, dt in spec:
                n = int(torch.tensor(shape).prod()) * torch.empty((), dtype=dt).element_size()
                views.append((name, shape, dt, off, n))
                off = (off + n + 15) // 16 * 16
            self._xdev = torch.empty(off, dtype=torch.uint8, device=self.device)
            self._xhost = torch.empty(off, dtype=torch.uint8).pin_memory()
            self._xviews = views
            self._xact_host = torch.empty(G, dtype=torch.int32).pin_memory()
            self._xact_dev = torch.empty(G, dtype=torch.int32, device=self.device)
            self._xd = {name: self._xdev[o:o + n].view(dt).view(shape) for name, shape, dt, o, n in views}
            self._xh = {name: self._xhost[o:o + n].view(dt).view(shape).numpy() for name, shape, dt, o, n in views}
        d = self._xd
        with torch.cuda.device(self.device):
            if ply_actions is not None:
                self._xact_host.numpy()[:] = ply_actions
                self._xact_dev.copy_(self._xact_host, non_blocking=True)
                check(self._lib.hexb_ply(self._h, _ptr(self._xact_dev), _ptr(d["ret"]), self._stream()))
            check(self._lib.hexb_export_state(self._h, *[_ptr(d[k]) for k in ("board", "regions", "region_counter", "cur", "done",
                                                                               "winner", "agent", "draws")], self._stream()))
        self._xhost.copy_(self._xdev, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return self._xh

    def state_dict(self):
        """Checkpoint of the whole shard: the packed device state (labels, records, statistics) plus the configuration it
        belongs to. The reference never saves env state (SURVEY.md section 5); this is the batched equivalent of pickling the env."""
        torch.cuda.current_stream(self.device).synchronize()
        off = self._state_ptr - self._state.data_ptr()
        cfg = {f[0]: getattr(self.cfg, f[0]) for f in self.cfg._fields_ if f[0] != "device"}
        sd = {"config": cfg, "layout_version": int(self._lib.hexb_version()), "state": self._state[off:off + self.state_bytes].clone()}
        # per-game bookkeeping that lives outside the packed blob: the pool opponent drawn at reset for the running episode, whose
        # turn it is, and (when enabled) the info-dict tensors
        for name in ("opp_index", "to_move", "eval_episode", "last_move_opponent", "winner"):
            t = getattr(self, name, None)
            if t is not None:
                sd[name] = t.clone()
        sd["opponent_eps"] = self.opponent_eps    # run-time switch of the handle (set_opponent_eps), not part of hexb_config
        return sd

    def load_state_dict(self, sd):
        cfg = {f[0]: getattr(self.cfg, f[0]) for f in self.cfg._fields_ if f[0] != "device"}
        if {k: v for k, v in sd["config"].items() if k != "eval_state"} != {k: v for k, v in cfg.items() if k != "eval_state"}:
            raise ValueError("checkpoint belongs to a different configuration: %r vs %r" % (sd["config"], cfg))
        if sd.get("layout_version") != int(self._lib.hexb_version()) or sd["state"].numel() != self.state_bytes:
            raise ValueError("checkpoint was written by another version of the packed state layout (%r, library %r)"
                             % (sd.get("layout_version"), int(self._lib.hexb_version())))
        off = self._state_ptr - self._state.data_ptr()
        self._state[off:off + self.state_bytes].copy_(sd["state"].to(self.device))
        if "eval_episode" in sd or bool(sd["config"].get("eval_state", 0)) != self.eval_state:   # set_eval is a run-time switch
            self.set_eval(bool(sd["config"].get("eval_state", 0)))
        if "opponent_eps" in sd and sd["opponent_eps"] != self.opponent_eps:   # HexEnv.eps of opponent_predict, a run-time switch too
            self.set_opponent_eps(sd["opponent_eps"])
        for name in ("opp_index", "to_move", "eval_episode", "last_move_opponent", "winner"):
            t = getattr(self, name, None)
            if t is not None:
                if name not in sd and name == "eval_episode":   # written before any set_eval call: no evaluation episode yet
                    t.zero_()
                    continue
                if name not in sd:
                    raise ValueError("checkpoint lacks %r, which this batch tracks" % name)
                t.copy_(sd[name].to(self.device))

    def import_boards(self, board_true, to_move=None, import_mask=None):
        """Overwrite games with preset positions (true coordinates, 0 BLACK / 1 WHITE / 2 EMPTY); labels are rebuilt in raster
        order like HexGame.__init__ does. On an env handle this is reset(sample_board=True) for the masked games."""
        b = self._in(board_true, (self.G, self.N, self.N), torch.int8, "board_true")
        tm = self._in(to_move, (self.G,), torch.int8, "to_move")
        im = self._in(import_mask, (self.G,), torch.uint8, "import_mask")
        with torch.cuda.device(self.device):
            check(self._lib.hexb_import_boards(self._h, _ptr(b), _ptr(tm), _ptr(im), self._stream()))

    def import_labels(self, board_true, regions, to_move=None, import_mask=None):
        """Overwrite games with preset positions AND their region-label planes (u8[G,2,N+2,N+2], the reference's layout), adopted
        as they are with region_counter = max(plane) + 1: HexGame.__init__(connected_stones=...)."""
        b = self._in(board_true, (self.G, self.N, self.N), torch.int8, "board_true")
        r = self._in(regions, (self.G, 2, self.N + 2, self.N + 2), torch.uint8, "regions")
        tm = self._in(to_move, (self.G,), torch.int8, "to_move")
        im = self._in(import_mask, (self.G,), torch.uint8, "import_mask")
        with torch.cuda.device(self.device):
            check(self._lib.hexb_import_labels(self._h, _ptr(b), _ptr(r), _ptr(tm), _ptr(im), self._stream()))

    # ------------------------------------------------------------------ tree search
    def copy_games(self, src, src_index=None, dst_index=None):
        """copy.deepcopy(env.simulator) for many games: game dst_index[i] of this RAW batch becomes a bare HexGame holding the
        position of game src_index[i] of `src` (any HexBatch of the same board size and variant on the same device), with the exact
        region counters; an env game whose agent is WHITE is converted to true coordinates. Indices are int64[count] (None = the
        identity; count = the length of a given index, else min of the two batch sizes); dst_index entries must be distinct and, when
        src is self, disjoint from the src games. Out-of-range pairs write nothing; games not named are untouched."""
        if not self.raw:
            raise ValueError("copy_games writes into a raw HexBatch (bare HexGame games)")
        if not isinstance(src, HexBatch) or src.N != self.N or src.variant != self.variant or src.device != self.device:
            raise ValueError("copy_games: src must be a HexBatch with the same board size and variant on %s" % self.device)
        lens = [int(torch.as_tensor(x).numel()) for x in (src_index, dst_index) if x is not None]
        if len(set(lens)) > 1:
            raise ValueError("src_index and dst_index must have the same length, got %s" % lens)
        count = lens[0] if lens else min(self.G, src.G)
        si = self._in(src_index, (count,), torch.int64, "src_index")
        di = self._in(dst_index, (count,), torch.int64, "dst_index")
        with torch.cuda.device(self.device):
            check(self._lib.hexb_copy_games(self._h, src._h, _ptr(si), _ptr(di), count, self._stream()))

    def playouts(self, num_playouts, first_playout=0, game_mask=None, out=None):
        """num_playouts random playouts per game from its current position (random_policy for both sides, filled to the end);
        returns int32[G]: playouts won by the side to move, -1 for finished, never-reset and masked-off (game_mask u8[G] == 0)
        games. Playout p uses its own stream (Philox counter c3 = p + 1), p in [first_playout, first_playout + num_playouts)."""
        num_playouts, first_playout = int(num_playouts), int(first_playout)
        if num_playouts < 1 or first_playout < 0 or first_playout + num_playouts >= 1 << 32:
            raise ValueError("need num_playouts >= 1, first_playout >= 0 and first_playout + num_playouts < 2**32")
        gm = self._in(game_mask, (self.G,), torch.uint8, "game_mask")
        out = self._chk(out, (self.G,), torch.int32, "out") if out is not None else torch.empty(self.G, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_playouts(self._h, num_playouts, first_playout, _ptr(gm), _ptr(out), self._stream()))
        return out

    def opponent_catch_up(self):
        """Let the built-in random opponent move in every game where it is to move (after import_boards on an env handle):
        SelfPlayEnv.reset -> continue_game (SelfplayWrapper.py:79-80)."""
        with torch.cuda.device(self.device):
            check(self._lib.hexb_half_step(self._h, 1, None, None, None, None, self._stream()))

    def stats(self, out=None):
        """Episode statistics since creation as a device int64[8] tensor (see STAT_NAMES)."""
        out = self._chk(out, (8,), torch.int64, "out") if out is not None else torch.empty(8, dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.hexb_stats(self._h, _ptr(out), self._stream()))
        return out
