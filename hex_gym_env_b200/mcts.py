"""Batched Monte-Carlo tree search on the device: one PUCT tree per game of a HexBatch (include/hexb.h, hexb_mcts_*).

    env = HexBatch(11, 4096, raw=True)          # any handle: raw, variant A or variant B env
    ...                                         # put the root positions into env
    tree = MCTS(env, max_nodes=801)
    tree.reset()
    tree.search(800, 8)                         # fused form: 800 simulations with 8 playouts per leaf, one launch
    tree.search(800, 8, policy=PLAYOUT_BRIDGE)  # ... with playouts that save bridges (include/hexb.h, HEXB_PLAYOUT_BRIDGE)
    visits, q, value, nodes_used = tree.root()

    tree.reset()                                # split form: a policy / value network evaluates the leaves
    for _ in range(800):
        obs, mask, pending = tree.select()
        priors, values = net(obs, mask)         # f32[G,C], f32[G]; rows with pending == 0 are ignored
        tree.expand(priors, values)

    visits = tree.root()[0]
    env.ply(visits.argmax(1).int())             # play the move (raw handle; an env step adds the reply too)
    tree.advance()                              # keep the subtree under the position reached, then search on from it

Per-cell arrays use the batch's action convention for the side to move at that node (variant B: the mover's view), so for an
env root at the agent's turn `visits.argmax(1)` is an action for `env.step`.
"""
import ctypes

import torch

from ._native import check
from .batch import PLAYOUT_RANDOM, HexBatch, _playout_policy, _ptr


class MCTS(object):
    def __init__(self, batch, max_nodes, c_puct=1.25, fpu=0.0):
        if not isinstance(batch, HexBatch):
            raise ValueError("MCTS needs a HexBatch")
        max_nodes = int(max_nodes)
        if not 1 <= max_nodes <= 1 << 24:
            raise ValueError("max_nodes must be in [1, 2**24], got %d" % max_nodes)
        c_puct, fpu = float(c_puct), float(fpu)
        if c_puct != c_puct or fpu != fpu:
            raise ValueError("c_puct and fpu must not be NaN")
        self.batch, self.max_nodes, self.c_puct, self.fpu = batch, max_nodes, c_puct, fpu
        self.device = batch.device
        self._lib = batch._lib
        nbytes = ctypes.c_size_t(0)
        check(self._lib.hexb_mcts_tree_bytes(batch._h, max_nodes, ctypes.byref(nbytes)))
        self.tree_bytes = int(nbytes.value)
        self.tree = torch.empty(self.tree_bytes, dtype=torch.uint8, device=self.device)   # torch's blocks are 512-byte aligned
        G, N, C = batch.G, batch.N, batch.C
        self.leaf_obs = torch.zeros((G, N, N), dtype=batch.obs_dtype, device=self.device)
        self.leaf_mask = torch.zeros((G, C), dtype=torch.uint8, device=self.device)
        self.pending = torch.zeros(G, dtype=torch.uint8, device=self.device)
        self._ready = False

    def _args(self):
        if not self._ready:
            raise RuntimeError("MCTS: call reset() first")
        return self.batch._h, ctypes.c_void_p(self.tree.data_ptr()), self.tree_bytes

    def reset(self, root_mask=None, first_playout=0):
        """A new tree on every root's current position; roots that are finished, never reset or have root_mask[g] == 0 stay
        inactive. Playout j of simulation s (fused form) is playout index first_playout + s * P + j of hexb_playouts."""
        first_playout = int(first_playout)
        if not 0 <= first_playout < 1 << 32:
            raise ValueError("first_playout must be in [0, 2**32)")
        rm = self.batch._in(root_mask, (self.batch.G,), torch.uint8, "root_mask")
        with torch.cuda.device(self.device):
            check(self._lib.hexb_mcts_init(self.batch._h, ctypes.c_void_p(self.tree.data_ptr()), self.tree_bytes, self.max_nodes,
                                           self.c_puct, self.fpu, first_playout, _ptr(rm), self.batch._stream()))
        self._ready = True

    def search(self, num_simulations, playouts_per_leaf, policy=PLAYOUT_RANDOM):
        """num_simulations simulations for every active root with playouts_per_leaf playouts per leaf, in one launch. policy:
        PLAYOUT_RANDOM (uniform random playouts) or PLAYOUT_BRIDGE (playouts that save bridges; a leaf's first ply may answer the
        move into the leaf). The policy belongs to the call, not to the tree: search(a) then search(b) equals search(a + b)
        under one policy."""
        num_simulations, playouts_per_leaf = int(num_simulations), int(playouts_per_leaf)
        if not (1 <= num_simulations < 1 << 31 and 1 <= playouts_per_leaf <= 1 << 16):
            raise ValueError("need num_simulations >= 1 and 1 <= playouts_per_leaf <= 65536")
        policy = _playout_policy(policy)
        h, t, nb = self._args()
        with torch.cuda.device(self.device):
            check(self._lib.hexb_mcts_search_policy(h, t, nb, num_simulations, playouts_per_leaf, policy, self.batch._stream()))

    def select(self):
        """Step 1 of one simulation: (leaf_obs [G,N,N] obs_dtype, leaf_mask u8[G,C], pending u8[G]), encode(view 1) of each pending
        root's leaf. Rows with pending == 0 (terminal leaf, already backed up, or inactive root) are not written. The tensors are
        owned by this object and rewritten by the next select."""
        h, t, nb = self._args()
        with torch.cuda.device(self.device):
            check(self._lib.hexb_mcts_select(h, t, nb, _ptr(self.leaf_obs), _ptr(self.leaf_mask), _ptr(self.pending),
                                             self.batch._stream()))
        return self.leaf_obs, self.leaf_mask, self.pending

    def expand(self, priors, values):
        """Steps 2-4 for the pending roots: priors f32[G,C] in the leaf mover's action order (cells not empty are ignored, nothing
        is renormalised), values f32[G] for the leaf's side to move."""
        G, C = self.batch.G, self.batch.C
        p = self.batch._in(priors, (G, C), torch.float32, "priors")
        v = self.batch._in(values, (G,), torch.float32, "values")
        h, t, nb = self._args()
        with torch.cuda.device(self.device):
            check(self._lib.hexb_mcts_expand(h, t, nb, _ptr(p), _ptr(v), self.batch._stream()))

    def advance(self, root_mask=None, first_playout=0):
        """Keep each root's subtree under the position its game has reached since the last reset / advance (one or two stones
        on along explored moves: a ply, or an env step with the opponent's reply), or start a fresh tree there as reset() would.
        Roots that are finished, never reset or have root_mask[g] == 0 become inactive. The kept root's counters are those of
        the edge into it; later fused simulations use playout indices from first_playout (include/hexb.h, hexb_mcts_advance)."""
        first_playout = int(first_playout)
        if not 0 <= first_playout < 1 << 32:
            raise ValueError("first_playout must be in [0, 2**32)")
        rm = self.batch._in(root_mask, (self.batch.G,), torch.uint8, "root_mask")
        h, t, nb = self._args()
        with torch.cuda.device(self.device):
            check(self._lib.hexb_mcts_advance(h, t, nb, first_playout, _ptr(rm), self.batch._stream()))

    def root(self):
        """(visits i32[G,C], q f32[G,C], value f32[G], nodes_used i32[G]) of every root; nodes_used == 0 marks an inactive root."""
        G, C = self.batch.G, self.batch.C
        visits = torch.empty((G, C), dtype=torch.int32, device=self.device)
        q = torch.empty((G, C), dtype=torch.float32, device=self.device)
        value = torch.empty(G, dtype=torch.float32, device=self.device)
        used = torch.empty(G, dtype=torch.int32, device=self.device)
        h, t, nb = self._args()
        with torch.cuda.device(self.device):
            check(self._lib.hexb_mcts_root(h, t, nb, _ptr(visits), _ptr(q), _ptr(value), _ptr(used), self.batch._stream()))
        return visits, q, value, used
