import json, os, sys
sys.path.insert(0, os.getcwd())
import torch
from hex_gym_env_b200 import HexBatch, VARIANT_B, AGENT_RANDOM
from bench import capture_steps
dev = torch.device("cuda", 0)
for N, G, K in ((19, 1 << 20, 40), (15, 1 << 20, 60), (13, 1 << 20, 60)):
    for form in (0, 1, 4):
        env = HexBatch(N, G, variant=VARIANT_B, device=0, seed=0, agent_mode=AGENT_RANDOM)
        if form: env.set_launch_form(form)
        env.reset(); env.rollout(400, outputs=False)
        for _ in range(3): env.step()
        g = capture_steps(env, dev, K); g.replay(); torch.cuda.synchronize()
        ts = []
        for rep in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(1e3 * e0.elapsed_time(e1) / K)
        print(json.dumps({"N": N, "G": G, "form": form, "us_min": round(min(ts), 1), "us_med": round(sorted(ts)[2], 1)}), flush=True)
        env.close(); del env, g
