"""TEST INFRASTRUCTURE ONLY - restatement of the playout policies of hexb_playouts_policy and hexb_mcts_search_policy
(include/hexb.h, HEXB_PLAYOUT_*) in plain Python, on top of the playout and tree-search oracles (oracle/playout.py,
oracle/mcts.py), which it leaves as they are.

PLAYOUT_RANDOM is oracle/playout.py's playout. PLAYOUT_BRIDGE plays the same plies with the same draws u: at ply k with mover m and
prev the cell of ply k-1, the reply set R is every cell e = prev + D[i] that is on the board and empty and whose prev + D[i-1] and
prev + D[i+1] are both m's (a stone of m, or an off-board point of m's edges). If R is not empty the ply plays its int(u * |R|)-th
cell in true row-major order, otherwise the int(u * n_empty)-th empty cell. Ply 0's prev is given by the caller (None = none).
"""
import numpy as np

from oracle import mcts, playout

BLACK, WHITE, EMPTY = playout.BLACK, playout.WHITE, playout.EMPTY
PLAYOUT_RANDOM, PLAYOUT_BRIDGE = 0, 1
D = ((-1, 0), (-1, 1), (0, 1), (1, 0), (1, -1), (0, -1))   # the six neighbours (dy, dx) in cyclic order


def owns(board, colour, y, x):
    """Is point (y, x) colour's: a stone of it on the board, or off the board on its side (BLACK beyond rows 0 and N-1, WHITE
    beyond columns 0 and N-1, corners nobody's)."""
    N = board.shape[0]
    if 0 <= y < N and 0 <= x < N:
        return board[y, x] == colour
    if colour == BLACK:
        return (y < 0 or y >= N) and 0 <= x < N
    return (x < 0 or x >= N) and 0 <= y < N


def bridge_replies(board, mover, prev):
    """The reply set of `mover` to the move at true cell `prev` (None = the empty set), in true row-major order."""
    if prev is None:
        return []
    N = board.shape[0]
    py, px = divmod(int(prev), N)
    out = []
    for i, (dy, dx) in enumerate(D):
        y, x = py + dy, px + dx
        if not (0 <= y < N and 0 <= x < N) or board[y, x] != EMPTY:
            continue
        (ay, ax), (by, bx) = D[i - 1], D[(i + 1) % 6]
        if owns(board, mover, py + ay, px + ax) and owns(board, mover, py + by, px + bx):
            out.append(y * N + x)
    return sorted(out)


def choice(u, n):
    """int(u * n), clamped to [0, n) (choice_of)."""
    return min(max(int(u * n), 0), n - 1)


def playout_plies(board, to_move, seed, game, p, policy=PLAYOUT_RANDOM, prev=None):
    """The plies of playout p: a list of (cell, u, reply set, random cell), where the random cell is the one PLAYOUT_RANDOM
    would play on the same board with the same u."""
    b = np.array(board, dtype=np.int8, copy=True)
    N = b.shape[0]
    empties = [int(c) for c in np.flatnonzero(b.reshape(-1) == EMPTY)]
    plies = []
    for k, u in enumerate(playout.draws(seed, game, p & 0xFFFFFFFF, len(empties))):
        mover = to_move if k % 2 == 0 else 1 - to_move
        replies = bridge_replies(b, mover, prev) if policy == PLAYOUT_BRIDGE else []
        rnd = empties[choice(u, len(empties))]
        c = replies[choice(u, len(replies))] if replies else rnd
        empties.remove(c)
        b[c // N, c % N] = mover
        plies.append((c, float(u), replies, rnd))
        prev = c
    return plies


def playout_winner(board, to_move, seed, game, p, policy=PLAYOUT_RANDOM, prev=None):
    """Winner (0 BLACK, 1 WHITE) of playout p and the cells it played."""
    b = np.array(board, dtype=np.int8, copy=True)
    N = b.shape[0]
    cells = [c for c, _, _, _ in playout_plies(b, to_move, seed, game, p, policy, prev)]
    for k, c in enumerate(cells):
        b[c // N, c % N] = to_move if k % 2 == 0 else 1 - to_move
    return (BLACK if playout.connects(b, BLACK) else WHITE), cells


def wins(board, to_move, seed, game, first_playout, num_playouts, policy=PLAYOUT_RANDOM, prev=None):
    """Playouts p in [first_playout, first_playout + num_playouts) (mod 2^32) won by `to_move`."""
    return sum(playout_winner(board, to_move, seed, game, p, policy, prev)[0] == to_move
               for p in range(first_playout, first_playout + num_playouts))


class RootTree(mcts.RootTree):
    """oracle/mcts.py's tree whose fused simulation takes a playout policy: a leaf at depth >= 1 gives its playouts the move into
    it as ply 0's prev; node 0 has none."""

    def simulate(self, P, policy=PLAYOUT_RANDOM):
        leaf = self.descend()
        v = mcts.F(-1)
        if not leaf["terminal"]:
            p0 = (self.first + self.s * P) & 0xFFFFFFFF
            prev = leaf["cell"] if leaf["depth"] >= 1 else None
            w = wins(leaf["board"].reshape(self.N, self.N), self.mover(leaf["depth"]), self.seed, self.gid, p0, P, policy, prev)
            v = mcts.F(2 * w - P) / mcts.F(P)
        if not (leaf["terminal"] and leaf["node"] >= 0):
            self.store(leaf)
        self.backup(leaf, v)
