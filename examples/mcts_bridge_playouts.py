"""MCTS valued by bridge-reply playouts (search(..., policy=PLAYOUT_BRIDGE)) against MCTS valued by uniform random playouts, at
the same simulations and playouts per move, all on the device.

G raw games (bare HexGame, variant B) start from the empty board. The bridge side plays BLACK in even games and WHITE in odd ones;
the random side plays the other colour. At every ply each side reset()s its tree on the games where it is to move, runs
search(S, P) with its playout policy and plays the most visited root cell (ply()). Each side's search time per move (the whole
batch's search call, CUDA events) is reported beside the result. Deterministic given the arguments. Results measured on a B200
are in profiles/g6_bridge_playouts.txt.

    python examples/mcts_bridge_playouts.py --board 11 --games 4096 --sims 200 --playouts 4
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


def run(board_size=7, games=4096, sims=200, playouts=4, c_puct=1.25, fpu=0.0, seed=0, device=0):
    import torch
    from hex_gym_env_b200 import MCTS, PLAYOUT_BRIDGE, PLAYOUT_RANDOM, VARIANT_B, HexBatch
    S, P = sims, playouts
    batch = HexBatch(board_size, games, variant=VARIANT_B, device=device, seed=seed, raw=True)
    batch.reset()
    dev, G, C = batch.device, batch.G, batch.C
    to_batch = lambda x: torch.from_numpy(x).to(dev)
    bridge_colour = np.arange(G) % 2
    sides = {"bridge": (MCTS(batch, max_nodes=S + 1, c_puct=c_puct, fpu=fpu), PLAYOUT_BRIDGE, 1 << 31),
             "random": (MCTS(batch, max_nodes=S + 1, c_puct=c_puct, fpu=fpu), PLAYOUT_RANDOM, 0)}
    ms = {k: [] for k in sides}
    winner = np.full(G, -1, np.int64)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for t in range(C):
        colour = t % 2                                              # every game starts with BLACK and alternates
        live = winner < 0
        a = np.full(G, -1, np.int64)
        for name, (tree, policy, base) in sides.items():
            mine = live & ((bridge_colour == colour) == (name == "bridge"))
            tree.reset(root_mask=to_batch(mine.astype(np.uint8)), first_playout=base + t * S * P)   # the streams never meet
            ev[0].record()
            tree.search(S, P, policy=policy)
            ev[1].record()
            ev[1].synchronize()
            if mine.any():
                ms[name].append(ev[0].elapsed_time(ev[1]))
            a = np.where(mine, tree.root()[0].argmax(1).cpu().numpy(), a)
        ret = batch.ply(to_batch(a.astype(np.int32))).cpu().numpy().astype(np.int64)   # -1: a finished game is left alone
        winner = np.where(live & ((ret == 0) | (ret == 1)), ret, winner)
    assert bool((winner >= 0).all()), "a game is still running after N*N plies"
    won = winner == bridge_colour
    k = int(won.sum())
    lo, hi = wilson(k, G)
    return dict(board=board_size, bridge_wins=k, games=G, win_rate=k / G, interval95=(lo, hi), sims=S, playouts=P,
                bridge_black_wins=int((won & (bridge_colour == 0)).sum()), bridge_white_wins=int((won & (bridge_colour == 1)).sum()),
                bridge_ms_per_move=float(np.mean(ms["bridge"])), random_ms_per_move=float(np.mean(ms["random"])),
                device_name=torch.cuda.get_device_name(dev))


def describe(r):
    return ("MCTS with bridge playouts vs MCTS with random playouts (%d sims x %d playouts per move each), %dx%d, %d games: bridge "
            "won %d (%.1f %%, 95 %% interval %.1f-%.1f %%; %d as BLACK, %d as WHITE); search time per move for the whole batch: "
            "bridge %.2f ms, random %.2f ms" % (r["sims"], r["playouts"], r["board"], r["board"], r["games"], r["bridge_wins"],
                                                100 * r["win_rate"], 100 * r["interval95"][0], 100 * r["interval95"][1],
                                                r["bridge_black_wins"], r["bridge_white_wins"], r["bridge_ms_per_move"],
                                                r["random_ms_per_move"]))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--board", type=int, default=7)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--playouts", type=int, default=4)
    ap.add_argument("--c-puct", type=float, default=1.25)
    ap.add_argument("--fpu", type=float, default=0.0)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    print(describe(run(a.board, a.games, a.sims, a.playouts, a.c_puct, a.fpu, a.seed)))


if __name__ == "__main__":
    main()
