"""Speed of the two playout policies (PLAYOUT_RANDOM, PLAYOUT_BRIDGE) on the GPU, timed in one run with the policies alternating
(CUDA events, after warm-up), with the card's name and power limit read in the same run. Writes one JSON document (default
profiles/g6_playout_policy_speed.json).

  playouts  4,096 mid-game 11x11 positions and 1,024 mid-game 19x19 positions (tools/search_speed.positions: variant B env games
            copied into a raw batch), 256 playouts each: playouts per second and plies per second (plies = empty cells x playouts)
  search    search(800, P) with max_nodes 801 from a fresh tree on the same kind of positions, P = 8 and 32: 4,096 roots at
            11x11 and 1,024 at 19x19; simulations per second and playouts per second (the tree is reset outside the timed window)
Each repetition times the random policy, then the bridge policy, on the same inputs; medians over the repetitions.

    python tools/playout_policy_speed.py [--out profiles/g6_playout_policy_speed.json] [--reps 7]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hex_gym_env_b200 import MCTS, PLAYOUT_BRIDGE, PLAYOUT_RANDOM  # noqa: E402
from search_speed import card, positions  # noqa: E402

POLICIES = (("random", PLAYOUT_RANDOM), ("bridge", PLAYOUT_BRIDGE))


def alternate(fns, reps, setup=None, warmup=2):
    """fns: {name: fn}. Each repetition runs setup() (untimed) and then times every fn in turn; medians per name."""
    for _ in range(warmup):
        for fn in fns.values():
            if setup:
                setup()
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for k, fn in fns.items():
            if setup:
                setup()
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[k].append(a.elapsed_time(b))
    out = {}
    for k, t in times.items():
        t.sort()
        out[k] = dict(median_ms=t[len(t) // 2], min_ms=t[0], max_ms=t[-1], reps=reps)
    return out


def playout_speed(N, G, P, reps):
    raw = positions(N, G, 2)
    outs = {k: torch.empty(G, dtype=torch.int32, device="cuda") for k, _ in POLICIES}
    t = alternate({k: (lambda k=k, pol=pol: raw.playouts(P, 0, out=outs[k], policy=pol)) for k, pol in POLICIES}, reps)
    ex = raw.export_state()
    live = ex["done"] == 0
    empties = int(((ex["regions"][:, :, 1:-1, 1:-1] == 0).all(1).sum((1, 2)) * live).sum())
    res = dict(board=N, positions=G, live_positions=int(live.sum()), playouts_per_position=P,
               mean_empty_cells=empties / max(int(live.sum()), 1))
    for k, _ in POLICIES:
        s = t[k]["median_ms"] * 1e-3
        w = outs[k][live]
        res[k] = dict(playouts_per_s=int(live.sum()) * P / s, plies_per_s=empties * P / s,
                      mean_win_share_side_to_move=float(w.float().mean()) / P, **t[k])
    res["bridge_time_over_random"] = t["bridge"]["median_ms"] / t["random"]["median_ms"]
    return res


def search_speed(N, G, S, P, reps):
    raw = positions(N, G, 3)
    tree = MCTS(raw, S + 1)
    t = alternate({k: (lambda pol=pol: tree.search(S, P, policy=pol)) for k, pol in POLICIES}, reps, setup=tree.reset)
    active = int((tree.root()[3] > 0).sum())
    res = dict(board=N, roots=G, active_roots=active, sims=S, playouts_per_leaf=P, max_nodes=S + 1)
    for k, _ in POLICIES:
        s = t[k]["median_ms"] * 1e-3
        res[k] = dict(sims_per_s=active * S / s, playouts_per_s=active * S * P / s, **t[k])
    res["bridge_time_over_random"] = t["bridge"]["median_ms"] / t["random"]["median_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "g6_playout_policy_speed.json"))
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("playout_policy_speed.py measures on the GPU; no CUDA device here")
    res = dict(card=card())
    res["playouts"] = [playout_speed(11, 4096, 256, a.reps), playout_speed(19, 1024, 256, a.reps)]
    res["search"] = [search_speed(N, G, 800, P, a.reps) for N, G in ((11, 4096), (19, 1024)) for P in (8, 32)]
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
