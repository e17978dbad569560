"""Step time of every launch form (1 / 4 warps per 32-game chunk, hexb_set_launch_form) on sub-wave and near-wave
batches, timed as ONE CUDA graph of K steps after a pre-roll (the same method as bench.py's extra_configs). One JSON line per
(config, form); `auto` is what the library picks by itself. Also times hexb_rollout (T steps per launch) per form."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from hex_gym_env_b200 import HexBatch, VARIANT_A, VARIANT_B, AGENT_RANDOM, AGENT_BLACK
from bench import moved_bytes, capture_steps

CONFIGS = [("6x6 4,096 (config 4 env side)", 6, 4096, VARIANT_B, AGENT_RANDOM),
           ("7x7 16,384", 7, 16384, VARIANT_A, AGENT_BLACK),
           ("7x7 65,536 (config 2)", 7, 65536, VARIANT_A, AGENT_BLACK),
           ("11x11 16,384", 11, 16384, VARIANT_B, AGENT_RANDOM),
           ("11x11 32,768", 11, 32768, VARIANT_B, AGENT_RANDOM),
           ("11x11 65,536", 11, 65536, VARIANT_B, AGENT_RANDOM),
           ("11x11 131,072 (config 3 shard)", 11, 131072, VARIANT_B, AGENT_RANDOM),
           ("19x19 16,384", 19, 16384, VARIANT_B, AGENT_RANDOM)]
K = 200
dev = torch.device("cuda", 0)
only = sys.argv[1:] 
for name, N, G, variant, am in CONFIGS:
    if only and not any(o in name for o in only):
        continue
    for form in (0, 1, 4):
        env = HexBatch(N, G, variant=variant, device=0, seed=0, agent_mode=am)
        env.set_launch_form(form)
        env.reset()
        env.rollout(300, outputs=False)
        for _ in range(3):
            env.step()
        g = capture_steps(env, dev, K)
        g.replay()
        torch.cuda.synchronize()
        best = 1e9
        for rep in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / K)
        # rollout: T steps per launch with outputs
        T = 32
        env.rollout(T)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            env.rollout(T)
        e1.record(); torch.cuda.synchronize()
        ro = e0.elapsed_time(e1) / (4 * T)
        print(json.dumps({"config": name, "board_size": N, "games": G, "form": form if form else "auto", "us_per_step": round(1e3 * best, 3),
                          "moved_GBps": round(G * moved_bytes(N) / (best * 1e-3) / 1e9, 1), "rollout_us_per_step": round(1e3 * ro, 3)}), flush=True)
        env.close(); del env, g
