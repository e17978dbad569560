"""TEST INFRASTRUCTURE ONLY - restatement of the playout definition of hexb_playouts (include/hexb.h).

Playout ``p`` of global game ``g`` starts from the true board with ``to_move`` (0 BLACK, 1 WHITE) first, colours alternating. Ply
``k`` draws ``u`` from Philox4x32-10 at counter ``(k, g_lo, g_hi, p + 1)`` under the seed, built into a double like every other
draw (``oracle/philox.py``), and plays the ``int(u * n_empty)``-th empty cell in true row-major order (``random_policy``,
minihex/__init__.py:8-12). The board is filled to the end; the winner is the colour whose edges connect (BLACK rows 0 and N-1,
WHITE columns 0 and N-1) under the reference's neighbourhood: the 3x3 window minus (-1,-1) and (+1,+1).
"""
import numpy as np

from .philox import philox4x32_10

BLACK, WHITE, EMPTY = 0, 1, 2
NEIGHBOURS = ((-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0))


def draws(seed, game, p, n):
    """u for plies 0..n-1 of playout p of global game `game`."""
    k = np.arange(n, dtype=np.uint64)
    game, seed = int(game), int(seed) & 0xFFFFFFFFFFFFFFFF
    a, b, _, _ = philox4x32_10(k, game & 0xFFFFFFFF, game >> 32, (int(p) + 1) & 0xFFFFFFFF, seed & 0xFFFFFFFF, seed >> 32)
    return ((a >> np.uint32(5)).astype(np.float64) * 67108864.0 + (b >> np.uint32(6)).astype(np.float64)) / 9007199254740992.0


def playout_cells(board, to_move, seed, game, p):
    """The true row-major cells playout p plays, in order (every empty cell once)."""
    board = np.asarray(board)
    empties = [int(c) for c in np.flatnonzero(board.reshape(-1) == EMPTY)]
    cells = []
    for u in draws(seed, game, p, len(empties)):
        n = len(empties)
        k = min(max(int(u * n), 0), n - 1)
        cells.append(empties.pop(k))
    return cells


def connects(board, colour):
    """Does `colour` connect its two edges on `board` (N x N, true coordinates)?"""
    N = board.shape[0]
    start = [(0, x) for x in range(N)] if colour == BLACK else [(y, 0) for y in range(N)]
    seen = set((y, x) for y, x in start if board[y, x] == colour)
    stack = list(seen)
    while stack:
        y, x = stack.pop()
        if (y if colour == BLACK else x) == N - 1:
            return True
        for dy, dx in NEIGHBOURS:
            yy, xx = y + dy, x + dx
            if 0 <= yy < N and 0 <= xx < N and board[yy, xx] == colour and (yy, xx) not in seen:
                seen.add((yy, xx))
                stack.append((yy, xx))
    return False


def playout_winner(board, to_move, seed, game, p):
    """Winner (0 BLACK, 1 WHITE) of playout p and the cells it played."""
    b = np.array(board, dtype=np.int8, copy=True)
    N = b.shape[0]
    cells = playout_cells(b, to_move, seed, game, p)
    for k, c in enumerate(cells):
        b[c // N, c % N] = to_move if k % 2 == 0 else 1 - to_move
    return (BLACK if connects(b, BLACK) else WHITE), cells


def wins(board, to_move, seed, game, first_playout, num_playouts):
    """Playouts p in [first_playout, first_playout + num_playouts) won by `to_move`."""
    return sum(playout_winner(board, to_move, seed, game, p)[0] == to_move
               for p in range(first_playout, first_playout + num_playouts))


class RawGame(object):
    """A bare HexGame rebuilt from exported state (regions f64[2,N+2,N+2], region_counter, cur, done, winner) with the counters
    as they are - what copy.deepcopy(env.simulator) holds - and make_move in TRUE coordinates (flood_fill HexGame.py:124-142,
    win check :102 / :111). Returns -1 (None), the winning colour, or 3 for an occupied or out-of-range cell (state untouched)."""

    def __init__(self, regions, region_counter, cur, done=0, winner=-1):
        self.regions = np.array(regions, dtype=np.int64, copy=True)
        self.counter = [int(region_counter[0]), int(region_counter[1])]
        self.cur, self.done, self.winner = int(cur), int(done), int(winner)
        self.N = self.regions.shape[1] - 2

    def make_move(self, cell):
        N = self.N
        if not 0 <= cell < N * N:
            return 3
        y, x = cell // N + 1, cell % N + 1
        if self.regions[0, y, x] or self.regions[1, y, x]:
            return 3
        reg = self.regions[self.cur]
        win = reg[y - 1:y + 2, x - 1:x + 2].copy()
        win[0, 0] = win[2, 2] = 0
        labels = sorted(set(int(v) for v in win.reshape(-1)) - {0})
        if not labels:
            reg[y, x] = self.counter[self.cur]
            self.counter[self.cur] += 1
        else:
            reg[y, x] = labels[0]
            for lab in labels[1:]:
                reg[reg == lab] = labels[0]
        ret = -1
        if reg[-1, -1] == 1:
            self.done, self.winner, ret = 1, self.cur, self.cur
        self.cur ^= 1
        return ret
