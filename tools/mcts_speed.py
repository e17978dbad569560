"""Speed of the batched tree search on the GPU (CUDA events, after warm-up), with the card's name and power limit read in the same
run. Writes one JSON document (default profiles/g2_mcts_speed.json).

  fused search   MCTS.search(S = 800, P) from pre-rolled positions (variant B env games, random agent colours, auto-reset, N*N/4
                 env steps, copied into a raw batch): 4,096 roots at 11x11 for P in {1, 8, 32}, 1,024 roots at 19x19 for P in
                 {1, 8}. Simulations per second (active roots x S) and playouts per second (x P). Each timed call starts from a
                 fresh tree (reset is outside the timed window).
  split round    one select -> expand round at 4,096 roots, 11x11, with a fixed torch "network" in between (uniform priors, zero
                 values), eager and replayed as a CUDA graph; the tree is reset before each block of rounds.
  tree bytes     hexb_mcts_tree_bytes for each configuration (max_nodes = S + 1).

    python tools/mcts_speed.py [--out profiles/g2_mcts_speed.json] [--reps 5]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hex_gym_env_b200 import MCTS  # noqa: E402
from search_speed import card, positions  # noqa: E402


def fused(N, G, S, P, reps):
    raw = positions(N, G, 3)
    tree = MCTS(raw, S + 1)
    times = []
    for i in range(reps + 1):
        tree.reset(first_playout=i * S * P)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tree.search(S, P)
        b.record()
        b.synchronize()
        if i:                                                     # the first call loads the module
            times.append(a.elapsed_time(b))
    times.sort()
    active = int((tree.root()[3] > 0).sum())
    s = times[len(times) // 2] * 1e-3
    return dict(board=N, roots=G, active_roots=active, sims=S, playouts_per_leaf=P, tree_bytes=tree.tree_bytes,
                median_ms=times[len(times) // 2], min_ms=times[0], max_ms=times[-1], reps=reps,
                sims_per_s=active * S / s, playouts_per_s=active * S * P / s)


def split(N, G, rounds, reps):
    raw = positions(N, G, 4)
    tree = MCTS(raw, rounds + 1)
    C = N * N
    priors = torch.empty(G, C, device="cuda")
    values = torch.empty(G, device="cuda")

    def round_():
        obs, mask, pending = tree.select()
        priors.copy_(mask.float() / mask.float().sum(1, keepdim=True).clamp_min(1))   # the fixed "network": uniform over legal cells
        values.zero_()
        tree.expand(priors, values)

    out = dict(board=N, roots=G, rounds=rounds, tree_bytes=tree.tree_bytes)
    tree.reset()
    round_()                                                      # load the modules
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        tree.reset()
        with torch.cuda.graph(graph, stream=s):
            round_()
    torch.cuda.current_stream().wait_stream(s)
    for name, fn in (("eager", round_), ("graph", graph.replay)):
        per = []
        for _ in range(reps):
            tree.reset()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(rounds):
                fn()
            b.record()
            b.synchronize()
            per.append(a.elapsed_time(b) * 1e3 / rounds)
        per.sort()
        out[name + "_us_per_round"] = per[len(per) // 2]
        out[name + "_us_per_round_min_max"] = [per[0], per[-1]]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "g2_mcts_speed.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mcts_speed.py measures on the GPU; no CUDA device here")
    res = dict(card=card())
    res["fused"] = [fused(11, 4096, 800, P, a.reps) for P in (1, 8, 32)] + [fused(19, 1024, 800, P, a.reps) for P in (1, 8)]
    res["split"] = split(11, 4096, 200, a.reps)
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
