"""MCTS that keeps its trees across moves (MCTS.advance) against MCTS that starts every move from a fresh tree (MCTS.reset), at
the same simulations per move, all on the device.

G raw games (bare HexGame, variant B) start from the empty board. The reusing side plays BLACK in even games and WHITE in odd
ones; the resetting side plays the other colour. At every ply both sides run MCTS.search(S, P) on the games where they are to move
and play the most visited root cell (ply()). Before its search
  reuse  advance()s its trees: the subtree under its own last move and the reply is kept, visits and values included,
  fresh  reset()s its trees on the new positions.
A search runs on every active root, so the reusing side keeps one MCTS object per colour it plays: each is advanced and searched
only at the plies where that colour is to move, and sees two stones on (its move and the reply) between calls.
Deterministic given the arguments. Measured on an NVIDIA B200 at a 1,000 W power limit, 7x7, 4,096 games, 4 playouts per leaf
(profiles/g5_mcts_reuse.txt): with 64 simulations per move the reusing side wins 2,167 games (52.9 %, 95 % interval 51.4-54.4 %),
with 200 it wins 2,132 (52.1 %, 50.5-53.6 %).

    python examples/mcts_reuse.py --board 7 --games 4096 --sims 64 --playouts 4
"""
import argparse
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def wilson(k, n, z=1.96):
    """95 % Wilson score interval of a binomial proportion k / n."""
    if n == 0:
        return 0.0, 1.0
    p = k / n
    d = 1 + z * z / n
    c = (p + z * z / (2 * n)) / d
    h = z * math.sqrt(p * (1 - p) / n + z * z / (4 * n * n)) / d
    return c - h, c + h


def play(games, new_tree, sims, playouts, to_batch, to_host):
    """Play every game of `games` (a raw batch at the empty board) to the end. new_tree(): a new MCTS on it; to_batch / to_host
    move numpy arrays to and from the batch's side. Returns (winner i64[G], the reusing side's colour i64[G], mean simulations
    an advanced root already held before its search)."""
    G, C, S, P = games.G, games.C, sims, playouts
    reuse_colour = np.arange(G) % 2
    reuse, fresh = [new_tree(), new_tree()], new_tree()
    started = [False, False]
    winner = np.full(G, -1, np.int64)
    held, advanced = 0, 0
    for t in range(C):
        colour = t % 2                                              # every game starts with BLACK and alternates
        live = winner < 0
        mine = (reuse_colour == colour) & live
        theirs = (reuse_colour != colour) & live
        tree = reuse[colour]
        first = (1 << 31) + t * (C + 1) * S * P                     # the two sides' playout streams never meet
        if started[colour]:
            tree.advance(root_mask=to_batch(mine.astype(np.uint8)), first_playout=first)
            visits = to_host(tree.root()[0]).astype(np.int64)
            held += int(visits.sum(1)[mine].sum())
            advanced += int(mine.sum())
        else:
            tree.reset(root_mask=to_batch(mine.astype(np.uint8)), first_playout=first)
            started[colour] = True
        tree.search(S, P)
        fresh.reset(root_mask=to_batch(theirs.astype(np.uint8)), first_playout=t * S * P)
        fresh.search(S, P)
        a = np.where(mine, to_host(tree.root()[0]).argmax(1), to_host(fresh.root()[0]).argmax(1))
        a = np.where(live, a, -1).astype(np.int32)                 # a finished game is left alone (-1: out of range, no change)
        ret = to_host(games.ply(to_batch(a))).astype(np.int64)
        winner = np.where(live & ((ret == 0) | (ret == 1)), ret, winner)
    assert bool((winner >= 0).all()), "a game is still running after N*N plies"
    return winner, reuse_colour, held / max(advanced, 1)


def summary(winner, reuse_colour, held, sims, playouts):
    G = len(winner)
    won = winner == reuse_colour
    k = int(won.sum())
    lo, hi = wilson(k, G)
    return dict(reuse_wins=k, games=G, win_rate=k / G, interval95=(lo, hi), sims=sims, playouts=playouts,
                reuse_black_wins=int((won & (reuse_colour == 0)).sum()), reuse_white_wins=int((won & (reuse_colour == 1)).sum()),
                mean_visits_kept=held)


def run(board_size=7, games=4096, sims=64, playouts=4, c_puct=1.25, fpu=0.0, seed=0, device=0):
    import torch
    from hex_gym_env_b200 import MCTS, VARIANT_B, HexBatch
    S, P = sims, playouts
    batch = HexBatch(board_size, games, variant=VARIANT_B, device=device, seed=seed, raw=True)
    batch.reset()
    dev = batch.device
    winner, colour, held = play(batch, lambda: MCTS(batch, max_nodes=2 * S + 1, c_puct=c_puct, fpu=fpu), S, P,
                                lambda x: torch.from_numpy(x).to(dev), lambda x: x.cpu().numpy())
    return summary(winner, colour, held, S, P)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--board", type=int, default=7)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=64)
    ap.add_argument("--playouts", type=int, default=4)
    ap.add_argument("--c-puct", type=float, default=1.25)
    ap.add_argument("--fpu", type=float, default=0.0)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    r = run(a.board, a.games, a.sims, a.playouts, a.c_puct, a.fpu, a.seed)
    print("MCTS with tree reuse vs MCTS with fresh trees (%d sims x %d playouts per move each), %dx%d, %d games: reuse won %d "
          "(%.1f %%, 95 %% interval %.1f-%.1f %%; %d as BLACK, %d as WHITE); an advanced root held %.1f visits before its search"
          % (r["sims"], r["playouts"], a.board, a.board, r["games"], r["reuse_wins"], 100 * r["win_rate"],
             100 * r["interval95"][0], 100 * r["interval95"][1], r["reuse_black_wins"], r["reuse_white_wins"], r["mean_visits_kept"]))


if __name__ == "__main__":
    main()
