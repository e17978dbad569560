"""Flat Monte-Carlo agent against the built-in random opponent, all on the device.

Every env step, for each of the G self-play games (variant B, agent colour drawn per game):
  1. copy every game's simulator into a raw children batch of G*C games (C = N*N: one child per action),
  2. play action a in child (g, a) - the agent's view is the mover's view in variant B, so a is passed unchanged; an occupied cell
     returns ret == 3 and that child is masked out,
  3. run P random playouts in every child; the child's value is P - wins (wins belong to the side to move there, the opponent),
     or P when the agent's ply already won,
  4. step the env with the best child's action.

    python examples/flat_mc.py --board 5 --games 1024 --playouts 32 --steps 200
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hex_gym_env_b200 import AGENT_RANDOM, VARIANT_B, HexBatch  # noqa: E402


def run(board_size=5, games=1024, playouts=32, steps=200, seed=0, device=0):
    N, G, C, P = board_size, games, board_size * board_size, playouts
    env = HexBatch(N, G, variant=VARIANT_B, device=device, seed=seed, agent_mode=AGENT_RANDOM, auto_reset=True)
    children = HexBatch(N, G * C, variant=VARIANT_B, device=device, seed=seed + 1, raw=True)
    dev = env.device
    roots = torch.arange(G, device=dev).repeat_interleave(C)
    actions = torch.arange(C, dtype=torch.int32, device=dev).repeat(G)
    env.reset()
    phases = ("copy", "ply", "playouts", "step")
    ms = dict.fromkeys(phases, 0.0)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)]
    for t in range(steps):
        ev[0].record()
        children.copy_games(env, roots)
        ev[1].record()
        ret = children.ply(actions)
        ev[2].record()
        wins = children.playouts(P, first_playout=t * P)
        ev[3].record()
        value = torch.where((ret == 0) | (ret == 1), float(P), (P - wins).float())   # the agent's ply won
        value = torch.where(ret == 3, float("-inf"), value).view(G, C)          # occupied cell
        env.step(actions=value.argmax(1).to(torch.int32))
        ev[4].record()
        torch.cuda.synchronize(dev)
        for i, k in enumerate(phases):
            ms[k] += ev[i].elapsed_time(ev[i + 1])
    st = env.stats().cpu().tolist()
    episodes, agent_wins = st[0], st[3]
    return dict(win_rate=agent_wins / max(episodes, 1), episodes=episodes, agent_wins=agent_wins, ms=ms)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--board", type=int, default=5)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--playouts", type=int, default=32)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    r = run(a.board, a.games, a.playouts, a.steps, a.seed)
    print("flat MC vs random, %dx%d, %d games, %d playouts per child: agent won %d of %d episodes (%.1f %%)"
          % (a.board, a.board, a.games, a.playouts, r["agent_wins"], r["episodes"], 100.0 * r["win_rate"]))
    print("time per step (ms): " + ", ".join("%s %.3f" % (k, v / a.steps) for k, v in r["ms"].items()))


if __name__ == "__main__":
    main()
