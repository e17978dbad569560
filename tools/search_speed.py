"""Speed of the tree-search primitives on the GPU (CUDA events, after warm-up), with the card's name and power limit read in the
same run. Writes one JSON document (default profiles/g1_search_speed.json).

  copy_games  4,096 roots broadcast into 121 children each at 11x11 (495,616 copies, 144 MB by the formula below; the 0.6 MB of
              roots are re-read from L2, the 72 MB of children are written):
              bytes moved per second, 2 * (C + 4 * (W + 2)) bytes per copied game (label bytes + record words, read and written)
  playouts    65,536 mid-game 11x11 positions x 256 playouts and 16,384 mid-game 19x19 positions x 256 playouts; the positions are
              pre-rolled env games (variant B, random agent colours, auto-reset) copied into a raw batch. Playouts per second and
              plies per second (plies = empty cells of the position x playouts: every playout fills the board)

    python tools/search_speed.py [--out profiles/g1_search_speed.json] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hex_gym_env_b200 import AGENT_RANDOM, VARIANT_B, HexBatch  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60).stdout.strip()
    except Exception as exc:   # the numbers are still measured; say why the card is unknown
        q = "nvidia-smi failed: %s" % exc
    return dict(name=torch.cuda.get_device_name(0), nvidia_smi=q)


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return dict(median_ms=times[len(times) // 2], min_ms=times[0], max_ms=times[-1], reps=reps)


def positions(N, G, seed):
    """G pre-rolled env games (N*N/4 env steps with auto-reset: every stage of a game) copied into a raw batch."""
    env = HexBatch(N, G, variant=VARIANT_B, device=0, seed=seed, agent_mode=AGENT_RANDOM, auto_reset=True)
    env.reset()
    env.rollout(N * N // 4, outputs=False)
    raw = HexBatch(N, G, variant=VARIANT_B, device=0, seed=seed, raw=True)
    raw.copy_games(env)
    return raw


def copy_speed(reps):
    N, roots, kids = 11, 4096, 121
    C, W = N * N, (N * N + 31) // 32
    src = positions(N, roots, 1)
    dst = HexBatch(N, roots * kids, variant=VARIANT_B, device=0, raw=True)
    idx = torch.arange(roots, device="cuda").repeat_interleave(kids)
    t = timed(lambda: dst.copy_games(src, idx), reps)
    nbytes = roots * kids * 2 * (C + 4 * (W + 2))
    return dict(board=N, roots=roots, children_per_root=kids, copies=roots * kids, bytes=nbytes,
                bytes_per_s=nbytes / (t["median_ms"] * 1e-3), **t)


def playout_speed(N, G, P, reps):
    raw = positions(N, G, 2)
    out = torch.empty(G, dtype=torch.int32, device="cuda")
    t = timed(lambda: raw.playouts(P, 0, out=out), reps)
    ex = raw.export_state()
    live = (ex["done"] == 0)
    empties = int(((ex["regions"][:, :, 1:-1, 1:-1] == 0).all(1).sum((1, 2)) * live).sum())
    s = t["median_ms"] * 1e-3
    return dict(board=N, positions=G, live_positions=int(live.sum()), playouts_per_position=P, mean_empty_cells=empties / max(int(live.sum()), 1),
                playouts_per_s=int(live.sum()) * P / s, plies_per_s=empties * P / s, **t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "g1_search_speed.json"))
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("search_speed.py measures on the GPU; no CUDA device here")
    res = dict(card=card(), copy_games=copy_speed(a.reps),
               playouts=[playout_speed(11, 65536, 256, a.reps), playout_speed(19, 16384, 256, a.reps)])
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
