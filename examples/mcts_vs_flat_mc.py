"""Batched MCTS against flat Monte-Carlo at an equal playout budget per move, all on the device.

G raw games (bare HexGame, variant B) start from the empty board. The MCTS agent plays BLACK in even games and WHITE in odd ones;
flat Monte-Carlo plays the other side. Every ply, in the games where it is to move:
  MCTS     MCTS.search(S, P) from the position (S * P playouts) and plays the most visited root cell,
  flat MC  copies the position into one child per cell, plays the cell and runs P' random playouts in each child (C * P' playouts,
           the child's value is P' - wins; a winning ply is worth P'), and plays the best child (examples/flat_mc.py).
Moves are applied with ply() until every game is over. Deterministic given the arguments.

    python examples/mcts_vs_flat_mc.py --board 5 --games 1024 --sims 200 --playouts 4
"""
import argparse
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hex_gym_env_b200 import MCTS, VARIANT_B, HexBatch  # noqa: E402


def wilson(k, n, z=1.96):
    """95 % Wilson score interval of a binomial proportion k / n."""
    if n == 0:
        return 0.0, 1.0
    p = k / n
    d = 1 + z * z / n
    c = (p + z * z / (2 * n)) / d
    h = z * math.sqrt(p * (1 - p) / n + z * z / (4 * n * n)) / d
    return c - h, c + h


def run(board_size=5, games=1024, sims=200, playouts=4, flat_playouts=None, c_puct=1.0, fpu=1.0, seed=0, device=0):
    N, G, C = board_size, games, board_size * board_size
    S, P = sims, playouts
    P_flat = flat_playouts or max(1, S * P // C)                # equal budget: C * P' = S * P
    games_ = HexBatch(N, G, variant=VARIANT_B, device=device, seed=seed, raw=True)
    games_.reset()
    dev = games_.device
    tree = MCTS(games_, max_nodes=S + 1, c_puct=c_puct, fpu=fpu)   # fpu 1: every cell is tried before any is revisited
    children = HexBatch(N, G * C, variant=VARIANT_B, device=device, seed=seed, raw=True)
    roots = torch.arange(G, device=dev).repeat_interleave(C)
    cells = torch.arange(C, dtype=torch.int32, device=dev).repeat(G)
    mcts_colour = torch.arange(G, device=dev) % 2                # 0 BLACK (even games), 1 WHITE (odd games)
    winner = torch.full((G,), -1, dtype=torch.int64, device=dev)
    for t in range(C):
        mcts_turn = (mcts_colour == t % 2)                        # every game starts with BLACK and alternates
        tree.reset(root_mask=mcts_turn.to(torch.uint8), first_playout=t * S * P)
        tree.search(S, P)
        visits = tree.root()[0]
        children.copy_games(games_, roots)
        ret = children.ply(cells)
        wins = children.playouts(P_flat, first_playout=t * P_flat)
        value = torch.where((ret == 0) | (ret == 1), float(P_flat), (P_flat - wins).float())
        value = torch.where(ret == 3, float("-inf"), value).view(G, C)
        actions = torch.where(mcts_turn, visits.argmax(1), value.argmax(1)).to(torch.int32)
        actions = torch.where(winner >= 0, -1, actions)            # a finished game is left alone (-1: out of range, no change)
        ret = games_.ply(actions).to(torch.int64)
        winner = torch.where((winner < 0) & ((ret == 0) | (ret == 1)), ret, winner)
    assert bool((winner >= 0).all()), "a game is still running after N*N plies"
    k = int((winner == mcts_colour).sum())
    lo, hi = wilson(k, G)
    return dict(mcts_wins=k, games=G, win_rate=k / G, interval95=(lo, hi), sims=S, playouts=P, flat_playouts=P_flat,
                mcts_black_wins=int(((winner == mcts_colour) & (mcts_colour == 0)).sum()),
                mcts_white_wins=int(((winner == mcts_colour) & (mcts_colour == 1)).sum()))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--board", type=int, default=5)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--playouts", type=int, default=4)
    ap.add_argument("--flat-playouts", type=int, default=None, help="default: sims * playouts / cells (equal budget)")
    ap.add_argument("--c-puct", type=float, default=1.0)
    ap.add_argument("--fpu", type=float, default=1.0)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    r = run(a.board, a.games, a.sims, a.playouts, a.flat_playouts, a.c_puct, a.fpu, a.seed)
    print("MCTS (%d sims x %d playouts) vs flat MC (%d playouts per cell), %dx%d, %d games: MCTS won %d (%.1f %%, 95 %% interval "
          "%.1f-%.1f %%; %d as BLACK, %d as WHITE)" % (r["sims"], r["playouts"], r["flat_playouts"], a.board, a.board, r["games"],
                                                      r["mcts_wins"], 100 * r["win_rate"], 100 * r["interval95"][0],
                                                      100 * r["interval95"][1], r["mcts_black_wins"], r["mcts_white_wins"]))


if __name__ == "__main__":
    main()
