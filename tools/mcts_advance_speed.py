"""Speed of tree reuse (MCTS.advance, hexb_mcts_advance) on the GPU (CUDA events, after warm-up), with the card's name and power
limit read in the same run. Writes one JSON document (default profiles/g5_mcts_advance_speed.json).

From pre-rolled positions (tools/search_speed.positions: variant B env games copied into a raw batch) every root runs
search(800, P) with max_nodes 801; the most visited root cell is played with ply(), and advance() re-roots every tree on it.
  4,096 roots at 11x11 and 1,024 roots at 19x19, P = 1.
  advance time: each timed call starts from a copy of the searched tree (the copy is outside the timed window).
  kept share: over the roots that stay active, the mean of (nodes used after) / (nodes used before) and of (simulations of the
              new root) / (simulations of the old root).

    python tools/mcts_advance_speed.py [--out profiles/g5_mcts_advance_speed.json] [--reps 9]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hex_gym_env_b200 import MCTS  # noqa: E402
from search_speed import card, positions  # noqa: E402


def advance(N, G, S, P, reps):
    raw = positions(N, G, 5)
    tree = MCTS(raw, S + 1)
    tree.reset()
    tree.search(S, P)
    visits, _, _, used0 = tree.root()
    sims0 = visits.sum(1) + 1                                     # Nn of the old root: every simulation but the first crossed an edge
    a = visits.argmax(1)
    kept_sims = visits.gather(1, a[:, None])[:, 0]
    snap = tree.tree.clone()
    raw.ply(torch.where(used0 > 0, a, -1).to(torch.int32))
    times = []
    for i in range(reps + 1):
        tree.tree.copy_(snap)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tree.advance(first_playout=S * P)
        e1.record()
        e1.synchronize()
        if i:                                                     # the first call loads the module
            times.append(e0.elapsed_time(e1))
    times.sort()
    v1, _, _, used1 = tree.root()
    on = (used0 > 0) & (used1 > 0)
    fresh = on & (used1 == 1) & (v1.sum(1) == 0)                  # the played move's child was never stored: a fresh tree
    kept_sims = torch.where(fresh, 0, kept_sims)
    return dict(board=N, roots=G, sims=S, playouts_per_leaf=P, max_nodes=S + 1, tree_bytes=tree.tree_bytes,
                active_after=int(on.sum()), fresh_after=int(fresh.sum()),
                median_ms=times[len(times) // 2], min_ms=times[0], max_ms=times[-1], reps=reps,
                mean_nodes_used_before=float(used0[on].float().mean()), mean_nodes_used_after=float(used1[on].float().mean()),
                mean_share_nodes_kept=float((used1[on].float() / used0[on].float()).mean()),
                mean_share_sims_kept=float((kept_sims[on].float() / sims0[on].float()).mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "g5_mcts_advance_speed.json"))
    ap.add_argument("--reps", type=int, default=9)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mcts_advance_speed.py measures on the GPU; no CUDA device here")
    res = dict(card=card())
    res["advance"] = [advance(11, 4096, 800, 1, a.reps), advance(19, 1024, 800, 1, a.reps)]
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
