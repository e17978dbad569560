"""TEST INFRASTRUCTURE ONLY - restatement of the tree search of hexb_mcts_* (include/hexb.h) in plain Python and numpy float32.

One ``RootTree`` per root game. Boards are true N x N arrays (0 BLACK, 1 WHITE, 2 EMPTY); per-cell arrays of a node are indexed by
the TRUE row-major cell, priors handed to ``expand`` by the action convention of a raw handle of the variant (variant B: the mover's
view, transposed for WHITE). Playouts are ``oracle/playout.py``'s. Every float is a numpy float32 and every operation rounds once,
as ``__fmul_rn`` / ``__fdiv_rn`` / ``__fadd_rn`` / ``__fsqrt_rn`` do on the device.
"""
import numpy as np

from . import playout

F = np.float32
EMPTY = 2
UNEXPANDED, EXPANDED, TERMINAL = 0, 1, 2


def action(variant, colour, N, c):
    """The per-cell index of true cell c for the side to move `colour`."""
    return c if variant == 0 or colour == 0 else (c % N) * N + c // N


def key(score, cell):
    """Order-preserving bits of the float32 score, ties to the lowest cell: the largest key wins."""
    b = int(np.array(score, np.float32).view(np.uint32))
    ordered = (~b & 0xFFFFFFFF) if b & 0x80000000 else (b | 0x80000000)
    return (ordered << 32) | (0xFFFFFFFF - cell)


class Node(object):
    def __init__(self, C, flag):
        self.flag, self.nn = flag, 0
        self.child = np.full(C, -1, np.int32)
        self.n = np.zeros(C, np.int32)
        self.w = np.zeros(C, np.float32)
        self.p = np.zeros(C, np.float32)


class RootTree(object):
    def __init__(self, board, to_move, max_nodes, c_puct, fpu, first_playout, variant=0, seed=0, gid=0):
        self.board = np.array(board, np.int8).reshape(-1)
        self.N = int(round(len(self.board) ** 0.5))
        self.C = len(self.board)
        self.t0, self.max_nodes, self.variant = int(to_move), int(max_nodes), int(variant)
        self.c_puct, self.fpu = F(c_puct), F(fpu)
        self.first, self.seed, self.gid = int(first_playout), int(seed), int(gid)
        self.nodes = [Node(self.C, UNEXPANDED)]
        self.s, self.vsum = 0, F(0)
        self.leaf = None

    def mover(self, depth):
        return self.t0 ^ (depth & 1)

    def best_cell(self, node, board):
        sq = np.sqrt(F(node.nn))
        best = 0
        for c in np.flatnonzero(board == EMPTY):
            n = int(node.n[c])
            q = node.w[c] / F(n) if n > 0 else self.fpu
            u = ((self.c_puct * node.p[c]) * sq) / F(1 + n)
            best = max(best, key(q + u, int(c)))
        return None if best == 0 else 0xFFFFFFFF - (best & 0xFFFFFFFF)

    def descend(self):
        """Step 1: the leaf (depth, node or -1, parent, cell), its board and the path's nodes and cells."""
        board = self.board.copy()
        path, cells = [0], [None]
        node, parent, cell, d = 0, -1, None, 0
        while d < self.C and self.nodes[node].flag == EXPANDED:
            c = self.best_cell(self.nodes[node], board)
            if c is None:
                break
            board[c] = self.mover(d)
            child = int(self.nodes[node].child[c])
            parent, cell, d = node, c, d + 1
            node = child
            path.append(node)
            cells.append(c)
            if node < 0 or self.nodes[node].flag == TERMINAL:
                break
        terminal = (node >= 0 and self.nodes[node].flag == TERMINAL) or \
            (node < 0 and playout.connects(board.reshape(self.N, self.N), self.mover(d - 1)))
        return dict(depth=d, node=node, parent=parent, cell=cell, board=board, path=path, cells=cells, terminal=terminal)

    def store(self, leaf, priors_true=None):
        """Step 3. priors_true: f32[C] by true cell (None = 1 / n_empty)."""
        node = leaf["node"]
        if node >= 0:
            if self.nodes[node].flag != UNEXPANDED:
                return
            target = self.nodes[node]
        else:
            if len(self.nodes) >= self.max_nodes:
                return
            leaf["path"][-1] = node = len(self.nodes)
            self.nodes[leaf["parent"]].child[leaf["cell"]] = node
            target = Node(self.C, UNEXPANDED)
            self.nodes.append(target)
        if leaf["terminal"]:
            target.flag = TERMINAL
            return
        target.flag = EXPANDED
        empty = leaf["board"] == EMPTY
        if priors_true is None:
            priors_true = np.full(self.C, F(1) / F(int(empty.sum())), np.float32)
        target.p[:] = np.where(empty, priors_true, F(0))

    def backup(self, leaf, v):
        """Step 4 with v for the leaf's side to move."""
        v, D = F(v), leaf["depth"]
        for d in range(D + 1):
            n = leaf["path"][d]
            if n >= 0:
                self.nodes[n].nn += 1
            if d >= 1:
                p, c = self.nodes[leaf["path"][d - 1]], leaf["cells"][d]
                p.n[c] += 1
                p.w[c] = p.w[c] + (v if (D - d) & 1 else -v)
        self.vsum = self.vsum + (-v if D & 1 else v)
        self.s += 1

    # ---- the two forms
    def simulate(self, P):
        """One simulation of hexb_mcts_search with P playouts per leaf."""
        leaf = self.descend()
        v = F(-1)
        if not leaf["terminal"]:
            p0 = (self.first + self.s * P) & 0xFFFFFFFF
            wins = playout.wins(leaf["board"].reshape(self.N, self.N), self.mover(leaf["depth"]), self.seed, self.gid, p0, P)
            v = F(2 * wins - P) / F(P)
        if not (leaf["terminal"] and leaf["node"] >= 0):
            self.store(leaf)
        self.backup(leaf, v)

    def select(self):
        """hexb_mcts_select for this root: the leaf's (obs i8[N,N], mask u8[C]) as encode(view 1) of a raw game, or None when the
        leaf was terminal and has been backed up."""
        leaf = self.descend()
        if leaf["terminal"]:
            if leaf["node"] < 0:
                self.store(leaf)
            self.backup(leaf, -1.0)
            return None
        self.leaf = leaf
        N, C, mover = self.N, self.C, self.mover(leaf["depth"])
        obs, mask = np.zeros(C, np.int8), np.zeros(C, np.uint8)
        for c in range(C):
            a, b = action(self.variant, mover, N, c), int(leaf["board"][c])
            mask[a] = b == EMPTY
            if self.variant == 0:
                obs[a] = b
            else:
                obs[a] = 0 if b == EMPTY else (-1 if b == mover else 1)
        return obs.reshape(N, N), mask

    def expand(self, priors, value):
        """hexb_mcts_expand for a pending root: priors f32[C] in the leaf mover's action order, value f32."""
        leaf, self.leaf = self.leaf, None
        mover = self.mover(leaf["depth"])
        pt = np.array([priors[action(self.variant, mover, self.N, c)] for c in range(self.C)], np.float32)
        self.store(leaf, pt)
        self.backup(leaf, value)

    def root(self):
        """(visits i32[C], q f32[C], value f32) in the root mover's action order."""
        visits, q = np.zeros(self.C, np.int32), np.zeros(self.C, np.float32)
        r = self.nodes[0]
        if r.flag == EXPANDED:
            for c in range(self.C):
                a = action(self.variant, self.t0, self.N, c)
                visits[a] = r.n[c]
                q[a] = r.w[c] / F(r.n[c]) if r.n[c] > 0 else F(0)
        value = self.vsum / F(r.nn) if r.nn > 0 else F(0)
        return visits, q, value
