#!/usr/bin/env python
"""bench.py - env-steps/s of 11x11 random self-play (BASELINE.json config 3) on N B200s, with the HBM roofline of the
fused step kernel and the CPU restatement of the reference loop timed beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path (one JSON line on rank 0)
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # the CPU reference arm (rank 0 only)

A "step" is one fused env step (agent ply + random-opponent reply + win check + reward/done + auto-reset + observation
and legal-action mask) over ALL games of the rank's shard: variant B (SelfPlayEnv + BaseRandomPolicy), agent colour
random per game, the agent itself a random policy drawing from the game's Philox stream ("random self-play").
Weak scaling: every GPU owns `--games-per-gpu` games (default 1,048,576 = config 3's one million games; at N GPUs the job
is N million games, sharded by global game index with no data-path collective; the only exchange is one NCCL all-reduce
of the int64[8] episode statistics, issued on a side stream AFTER the timed steps and timed on its own as collective_ms).

Order of the device-resident leg: reset -> [3 steps, then K steps timed = `early_game`] -> untimed pre-roll of --preroll steps
(one hexb_rollout launch: de-synchronises the games over a few ~54-step episodes so that the steady state is measured
whatever --warmup is) -> W warm-up steps -> the K steps captured as ONE CUDA graph, replayed once untimed -> barrier ->
e0 | one replay = exactly K step-kernel launches | e1 -> statistics + all-reduce on the side stream. `value` = all ranks' env
steps / max over ranks of [e0, e1] (`ms_per_rank` lists every rank's figure).

roofline: achieved = bytes this design must move per launch / the step kernel's average duration in that same bracket (it
holds nothing else), B'(N) = 2*(C + 4*(W+2)) + 2*C + 5 bytes per env step (packed state in and out, obs, mask, reward, done;
537 B at 11x11; DESIGN.md section 3). `frac_contract` is the same time against SURVEY.md 8(d)'s B(N) = 831 B, which assumes a
state twice as large as this design's and therefore exceeds 1.

e2e: the same step through hexb_step_host with pinned HOST buffers (actions H2D, obs/mask/reward/done D2H inside the timed
region). cpu_baseline / --impl reference: the UNMODIFIED reference's SelfPlayEnv loop from oracle/_ref (oracle/make_ref.py,
oracle/ref_loop.py), one process per host core. extra_configs (1-GPU line only): BASELINE configs 2 and 5, the literal
config-3 shard (131,072 games) and config 4's env side, each pre-rolled and timed the same way.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BOARD = 11
GAMES_PER_GPU = 1 << 20
METRIC = "env_steps_per_sec_11x11_random_selfplay"
UNIT = "env-steps/s"


def contract_bytes(N):
    """SURVEY.md section 8(d): B(N) = 4 + 2*S(N) + 2*C + 5, S(N) = 8W + 2C + 16 (algorithmic bytes per env-step per game)."""
    C = N * N
    W = (C + 31) // 32
    return 4 + 2 * (8 * W + 2 * C + 16) + 2 * C + 5


def moved_bytes(N, sampled=True):
    """Bytes this implementation really moves per env-step per game: packed state in + out (C label bytes + (W+2) u32
    record words), obs + mask + reward + done out (+ actions in when the agent is external)."""
    C = N * N
    W = (C + 31) // 32
    S = C + 4 * (W + 2)
    return 2 * S + 2 * C + 5 + (0 if sampled else 4)


class ClockSampler(object):
    """Samples SM clock + throttle reasons with NVML while the timed region runs."""

    BAD = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown"}
    NOTE = {0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks", 0x100: "display_clock", 0x10: "sync_boost"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as exc:  # no NVML: report that instead of inventing clocks
            self.nv, self.err = None, str(exc)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in list(self.BAD.items()) + list(self.NOTE.items()):
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.01)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml_unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------------- CPU legs
def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_port_rate(N, budget_s, threads):
    """The C restatement of the reference loop (oracle/hexref.c), `threads` pthreads over independent games."""
    from oracle import hexref
    hexref.set_threads(threads)
    G = 2048 * threads
    b = hexref.RefBatch(hexref.KIND_SELFPLAY_B, N, G, seed=0, agent_mode=2)
    b.reset()
    for _ in range(3):
        b.step()
    n, t0 = 0, time.perf_counter()
    while True:
        b.step()          # obs + mask + reward + done written every step, like the reference loop computes them
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s:
            break
    return G * n / dt, "%d games x %d steps (C port, %d threads)" % (G, n, threads)


def ref_kind():
    """"reference" when the byte-identical copy of the reference (oracle/_ref, oracle/make_ref.py) is present, else "port"."""
    from oracle import ref_loop
    return "reference" if ref_loop.available() else "port"


def py_rate(N, seconds, procs, kind):
    """The reference's random self-play loop in child interpreters (keeps fork() away from this process's CUDA context):
    kind "reference" = the UNMODIFIED minihex classes from oracle/_ref (oracle/ref_loop.py), "port" = the Python/numpy
    restatement (oracle/pyloop.py), used only when the copy is missing."""
    import subprocess
    mod = "oracle.ref_loop" if kind == "reference" else "oracle.pyloop"
    out = subprocess.run([sys.executable, "-m", mod, str(N), str(seconds), str(procs)], cwd=ROOT, check=True,
                         stdout=subprocess.PIPE, text=True, env=dict(os.environ, OMP_NUM_THREADS="1")).stdout
    j = json.loads(out.strip().splitlines()[-1])
    return j["value"], j["sample"]


def cpu_baseline(N, budget_s=12.0):
    cores, kind = host_cores(), ref_kind()
    v, sample = py_rate(N, budget_s, cores, kind)
    p1, _ = py_rate(N, min(budget_s, 3.0), 1, kind)
    out = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "one_core": p1}
    if kind == "reference":   # how the restatements compare with the real thing, same box, same run
        out["python_port_all_cores"], _ = py_rate(N, 3.0, cores, "port")
    out["c_port_1_thread"], _ = cpu_port_rate(N, 2.0, 1)
    out["c_port_all_threads"], _ = cpu_port_rate(N, 3.0, cores)
    return out


def workload_config(args, world):
    """The `config` object of the JSON line - the same for both arms (the reference arm samples this workload on host cores)."""
    N, G, K = args.board, args.games_per_gpu, args.steps
    use_graph = (not args.no_graph) and K >= 2
    return {"workload": ("11x11 SelfPlayEnv (variant B) random self-play, random opponent, auto-reset (BASELINE config 3)" if N == 11
                         else "%dx%d SelfPlayEnv random self-play" % (N, N)),
            "board_size": N, "games_per_gpu": G, "global_games": world * G, "parallelism": "games sharded by index x%d" % world,
            "l2_policy": "working set %.0f MB per step > 126 MB L2" % (G * moved_bytes(N) / 1e6),
            "device_memory": "packed state, obs and mask in compressible device memory (hexb_mem_alloc: cuMemCreate with "
                             "CU_MEM_ALLOCATION_COMP_GENERIC) when the state is at least 64 MiB; roofline.memory_kind says what was granted",
            "agent": "random policy (BaseRandomPolicy) drawing from the game's own stream", "seed": args.seed,
            "preroll_steps": args.preroll + (K if use_graph else 0),
            "launch": ("ONE CUDA graph of the K = %d step launches" % K) if use_graph else "one launch per step"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path - the UNMODIFIED minihex SelfPlayEnv loop
    (mask = legal_actions(); a = BaseRandomPolicy().choose_action(obs); step(a); reset on done) from oracle/_ref, one process
    per host core (the reference is single-threaded). Every "step" is one bounded sample of that loop on all cores; exactly
    --steps samples are timed after --warmup untimed ones, and the sample length is chosen so that the run ends in ~1 minute."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N = args.board
    cores, kind = host_cores(), ref_kind()
    steps, warm = max(args.steps, 1), max(args.warmup, 0)
    per_step_s = min(2.0, max(0.4, args.ref_budget / (steps + 0.5 * warm)))   # interpreter start-up (~0.3 s) comes on top of each
    for _ in range(warm):
        py_rate(N, 0.5 * per_step_s, cores, kind)
    t0 = time.perf_counter()
    samples = []
    for _ in range(steps):
        v, sample = py_rate(N, per_step_s, cores, kind)
        samples.append(v)
    dt = time.perf_counter() - t0
    v = sum(samples) / len(samples)
    c_all, c_sample = cpu_port_rate(N, 2.0, cores)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, max(args.gpus, 1)),
            "arm_note": "reference CPU loop, one env per host core (%d); each step = one %.2f s sample of the loop on every core; "
                        "the GPU-side keys of config describe the arm this one is compared with" % (cores, per_step_s),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": "%s, %d processes x %.2f s x %d steps"
                                       % ("unmodified minihex SelfPlayEnv loop (oracle/_ref)" if kind == "reference"
                                          else "python/numpy restatement of the minihex loop (oracle/_ref missing)", cores, per_step_s, steps),
                             "c_port_all_threads": c_all, "c_port_sample": c_sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=args.out, flush=True)


# ---------------------------------------------------------------------------------------------------- GPU arm
def pin_rank_cpus(local, local_world):
    """Give this rank its own slice of the host CPUs. NVML's ideal set for the GPU is the starting point (on these single-socket
    VMs it is the same 32 CPUs for every GPU, which is how 8 launch loops + 8 NVML samplers + the NCCL proxies ended up sharing
    cores in round 1); the ranks whose GPUs share a set split it evenly by position."""
    if not hasattr(os, "sched_getaffinity"):
        return "unchanged (no sched_getaffinity)"
    allowed = sorted(os.sched_getaffinity(0))
    mine, peers = allowed, list(range(local_world))
    try:
        import pynvml
        pynvml.nvmlInit()
        words = (max(allowed) // 64) + 1

        def ideal(i):
            m = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(i), words)
            s = [c for c in allowed if (m[c // 64] >> (c % 64)) & 1]
            return s or allowed
        sets = [ideal(i) for i in range(local_world)]
        mine = sets[local]
        peers = [i for i in range(local_world) if sets[i] == mine]
    except Exception:
        pass
    k, n = peers.index(local), len(peers)
    per = max(len(mine) // n, 1)
    sl = mine[k * per:(k + 1) * per] if k * per < len(mine) else mine
    try:
        os.sched_setaffinity(0, sl)
    except Exception as exc:
        return "not set (%s)" % (str(exc)[:60],)
    return "cpus %d-%d (%d of %d allowed, slice %d/%d)" % (sl[0], sl[-1], len(sl), len(allowed), k, n)


def capture_steps(env, dev, n, **kw):
    """n calls of env.step(**kw) as ONE CUDA graph (a replay = n step-kernel launches, no host work in between).
    g.outputs holds the tensors the last captured step writes."""
    import torch
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for _ in range(n):
                g.outputs = env.step(**kw)
    torch.cuda.current_stream(dev).wait_stream(side)
    return g


DUMP_BYTES = 48 << 20    # --dump-outputs: at most this much float32 in all


def dump_outputs(out_dir, step_out, G, game_offset, max_bytes=DUMP_BYTES):
    """Write the last timed step's outputs (obs, mask, reward, done: what env.step() returns) as float32 .npy files, for a
    fixed, seeded sample of the games that fits max_bytes, and the sample's global game indices as game_index.npy (float64)."""
    import numpy as np
    import torch
    per_game = sum(4 * (t[0].numel() if t.dim() > 1 else 1) for t in step_out.values()) + 8
    S = min(G, max_bytes // per_game)
    idx = np.sort(np.random.default_rng(0).choice(G, S, replace=False))
    rows = torch.from_numpy(idx).to(next(iter(step_out.values())).device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "game_index.npy"), (idx + game_offset).astype(np.float64))
    for name, t in step_out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, rows).to(torch.float32).cpu().numpy())


def time_steps(env, dev, K, use_graph, reps=1):
    """CUDA-event time (ms) of `reps` x K env.step() launches on the current stream; with a graph, one replay = K launches."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g = capture_steps(env, dev, K) if use_graph else None
    if g is not None:
        g.replay()                       # untimed: first replay of a fresh graph uploads it
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        if g is not None:
            g.replay()
        else:
            for _ in range(K):
                env.step()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1), (K if g is not None else 0)


def extra_config(name, N, G, variant, agent_mode, K, preroll, dev, peak):
    """One more BASELINE configuration on this GPU (N = 1 run only): untimed pre-roll, then K graph-replayed steps."""
    import torch
    from hex_gym_env_b200 import HexBatch
    env = HexBatch(N, G, variant=variant, device=dev.index, seed=0, agent_mode=agent_mode, auto_reset=True)
    env.reset()
    left = preroll
    while left > 0:                      # untimed, in launches of at most 1,000 steps
        env.rollout(min(left, 1000), outputs=False)
        left -= 1000
    for _ in range(3):
        env.step()
    ms, _ = time_steps(env, dev, K, True, reps=3)   # three replays of the K-step graph, timed as one bracket
    us = 1e3 * ms / (3 * K)
    mv = G * moved_bytes(N) / (us * 1e-6) / 1e9
    out = {"config": name, "board_size": N, "games": G, "steps": 3 * K, "preroll_steps": preroll, "us_per_step": us,
           "env_steps_per_sec": G / (us * 1e-6), "moved_GBps": mv, "frac_of_hbm_peak": mv / peak,
           "bytes_per_env_step_moved": moved_bytes(N), "memory_kind": env.memory_kind}
    env.close()
    del env
    torch.cuda.empty_cache()
    return out


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from hex_gym_env_b200 import HexBatch, VARIANT_A, VARIANT_B, AGENT_RANDOM, AGENT_BLACK

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.set_num_threads(1)     # host-side torch work here is a few scalar reads; idle OpenMP workers would spin on the cores the
                                 # library's own host threads (packed transport) run on
    numa = pin_rank_cpus(local, local_world)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N, G, K, Wm = args.board, args.games_per_gpu, args.steps, args.warmup
    use_graph = (not args.no_graph) and K >= 2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_ms(ms):
        if world == 1:
            return [ms]
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        out = torch.empty(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(out, t)
        return out.cpu().tolist()

    # ------------------------------------------------ device-resident leg (value + roofline)
    env = HexBatch(N, G, variant=VARIANT_B, device=local, seed=args.seed, game_offset=rank * G, agent_mode=AGENT_RANDOM,
                   auto_reset=True)
    main = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(device=dev)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    env.reset()
    # (a) the early game, for the record: all games start together on empty boards, few merges, no game ends
    for _ in range(3):
        env.step()
    early_ms, _ = time_steps(env, dev, K, use_graph)
    # (b) untimed, declared pre-roll: games de-synchronise over a few episodes (mean episode ~54 env steps at 11x11), so
    #     that the timed steps see the steady-state mix of merges, finished games and restarts whatever --warmup is
    env.rollout(args.preroll, outputs=False)
    for _ in range(Wm):
        env.step()
    graph = capture_steps(env, dev, K) if use_graph else None
    if graph is not None:
        graph.replay()                   # untimed: uploads the graph (K more steps of pre-roll)
    for _ in range(3):                   # the collective is warm before anything is timed
        env.stats(out=stats)
        if world > 1:
            dist.all_reduce(stats)
    s0 = stats.clone()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    e0.record()
    if graph is not None:
        graph.replay()                   # exactly K step launches
        last = graph.outputs
    else:
        for _ in range(K):
            last = env.step()
    e1.record()
    # K7 + the path's only collective (64 bytes), on a side stream that waits for the K steps: it is never between two step
    # kernels, and it is outside the [e0, e1] bracket (timed on its own as collective_ms)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        env.stats(out=stats)
        c0.record()
        if world > 1:
            dist.all_reduce(stats)
        c1.record()
    main.wait_stream(side)
    barrier()
    clocks = sampler.stop()
    my_ms = e0.elapsed_time(e1)
    per_rank = gather_ms(my_ms)
    ms = max(per_rank)
    collective_ms = c0.elapsed_time(c1) if world > 1 else 0.0
    launches = K
    value = world * G * K / (ms * 1e-3)
    ds = (stats - s0).cpu().tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, G, rank * G)

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    kern_ms = my_ms / K                  # the bracket holds nothing but the K step-kernel launches
    Bm, Bc = moved_bytes(N), contract_bytes(N)
    achieved = G * Bm / (kern_ms * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        ent = tj.get("N%d_G%d" % (N, G))
        if ent:
            traffic = ent["dram_bytes_per_launch"]
    except Exception:
        pass
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": "hexb_step_kernel<%d, KIND_STEP, %s>" % (N, "several-rows sweep" if (G + 127) // 128 * 4 <= sms * (28 if N <= 8 else 12) else "one-row sweep"),
                "kernel_ms": kern_ms, "bytes_per_env_step": Bm, "bytes_per_launch": G * Bm,
                "bytes_formula": "B'(N) = 2*(C + 4*(W+2)) [packed state in + out] + 2*C [obs + mask] + 5 [reward + done] (+4 with external actions); C = N*N, W = ceil(C/32)",
                "frac_contract": G * Bc / (kern_ms * 1e-3) / 1e9 / peak, "bytes_per_env_step_contract": Bc,
                "note": "achieved/frac count the bytes this design must move per env step (DESIGN.md section 3); frac_contract uses SURVEY "
                        "8(d)'s B(N), whose state term (290 B per game each way) is twice this design's 145 B and therefore exceeds 1. "
                        "20 MiB of the state stay L2-resident across steps and, in compressible memory (memory_kind), the L2's inline "
                        "compression shrinks what reaches HBM further, so HBM sees less than bytes_per_launch (traffic = ncu dram bytes "
                        "per launch)",
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                "memory_kind": env.memory_kind}
    early = {"ms_per_step": early_ms / K, "value": world * G * K / (early_ms * 1e-3),
             "note": "the same K steps timed right after reset (3 warm-up steps): every game in its opening, no merges, no restarts"}
    env.close()
    del env, graph
    torch.cuda.empty_cache()

    # ------------------------------------------------ end-to-end leg: host actions in, host obs/mask/reward/done out
    E = min(K, args.e2e_steps)
    Ew = 24    # untimed: the adaptive transport searches its split during the first 22 calls
    # (untimed) record a legal random trajectory on the device so that the timed loop replays HOST actions
    rec = HexBatch(N, G, variant=VARIANT_B, device=local, seed=args.seed + 1, game_offset=rank * G, agent_mode=AGENT_RANDOM,
                   auto_reset=True)
    rec.reset()
    host_actions = torch.empty((E + Ew, G), dtype=torch.int32).pin_memory()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    for t in range(E + Ew):
        u = torch.rand(G, dtype=torch.float64, device=dev, generator=gen)
        a = rec.sample_actions(u)
        host_actions[t].copy_(a)
        rec.step(a, outputs=False)
    torch.cuda.synchronize()
    rec.close()
    del rec
    def e2e_leg(mode):
        """E timed steps of the host-buffer call hexb_step_host. mode "adaptive" = the call as shipped (obs + mask of some games
        as plain DMA copies, of the others as 2 bits per cell expanded by host threads, the split found by timing a few candidates in the first 22 calls);
        "dma" = plain copies only (hexb_set_host_transport(1)); "packed" = 2-bit transport only (0)."""
        env = HexBatch(N, G, variant=VARIANT_B, device=local, seed=args.seed + 1, game_offset=rank * G, agent_mode=AGENT_RANDOM,
                       auto_reset=True)
        env.reset()
        if mode != "adaptive":
            env.set_host_transport(1.0 if mode == "dma" else 0.0)
        io = env.pinned_io()
        for t in range(Ew):
            env.step_host(host_actions[t], io)
        barrier()
        t0 = time.perf_counter()
        e0.record()
        checksum = 0.0
        for t in range(Ew, Ew + E):
            # this step's inputs are a row of pinned host memory; the call copies them to the device, steps, copies the results
            # back and returns with them in host memory
            env.step_host(host_actions[t], io)
            checksum += float(io["reward"][0]) + float(io["obs"][G - 1, N - 1, N - 1]) + float(io["mask"][G - 1, N * N - 1])   # host reads of the step's results
        e1.record()
        barrier()
        ms = max(gather_ms(e0.elapsed_time(e1)))
        wall_ms = (time.perf_counter() - t0) * 1e3
        invalid = int(env.stats().cpu()[5])
        f = env.host_transport()
        gd = int(f * G + 0.5) // 32 * 32 if f < 1.0 else G
        d2h = gd * 2 * N * N + ((G - gd) * N * N + 15) // 16 * 4 + 5 * G
        out = {"value": world * G * E / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 4 * G, "d2h_bytes_per_step": d2h, "steps": E,
               "ms_per_step": ms / E, "wall_ms_per_step": wall_ms / E,
               "api": "hexb_step_host (C ABI, pinned host buffers); transport %s: %.0f %% of the games' obs + mask as plain DMA, the rest as "
                      "2 bits per cell expanded by %d host threads" % (mode, 100.0 * gd / G, env._lib.hexb_host_threads()),
               "dma_fraction": f, "illegal_moves_in_replay": invalid, "cpu_affinity": numa, "checksum": checksum}
        env.close()
        del env
        torch.cuda.empty_cache()
        return out

    legs = {m: e2e_leg(m) for m in ("dma", "packed", "adaptive")}
    assert len({legs[m]["checksum"] for m in legs}) == 1, "the host transports returned different results"
    e2e = dict(legs["adaptive"])         # the headline end-to-end number: the public call as shipped
    for m in ("dma", "packed"):
        e2e[m + "_only"] = {k: legs[m][k] for k in ("value", "ms_per_step", "d2h_bytes_per_step")}
    launches_e2e = 2 * E

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args, world),
            "roofline": roofline, "e2e": e2e, "gpu_launches": launches,
            "gpu_launches_detail": {"timed_region": "%d x hexb_step_kernel" % K, "after_timed_region": "1 x hexb_stats_kernel%s (side stream)" % (" + ncclAllReduce int64[8]" if world > 1 else ""), "e2e_region": launches_e2e},
            "ms_per_rank": [m / K for m in per_rank], "collective_ms": collective_ms, "clocks": clocks, "early_game": early,
            "plies_per_sec": ds[7] / (ms * 1e-3), "episodes_in_timed_region": ds[0],
            "episode_stats": dict(zip(("episodes", "black_wins", "white_wins", "agent_wins", "episode_plies", "invalid_ends",
                                       "env_steps", "plies"), ds))}
    if rank == 0 and world == 1 and not args.no_extra:
        # the other BASELINE configurations that fit one GPU, and the literal config-3 shard (1 Mi games over 8 GPUs)
        line["extra_configs"] = [
            extra_config("config 2: 7x7 HexEnv (variant A) + random_policy opponent, 65,536 games", 7, 65536, VARIANT_A, AGENT_BLACK, 200, 100, dev, peak),
            extra_config("config 3 shard: 11x11 SelfPlayEnv, 131,072 games (1 Mi games / 8 GPUs)", 11, 131072, VARIANT_B, AGENT_RANDOM, 200, 300, dev, peak),
            extra_config("config 4 env side: 6x6 SelfPlayEnv, 4,096 games", 6, 4096, VARIANT_B, AGENT_RANDOM, 200, 100, dev, peak),
            extra_config("config 5: 19x19 SelfPlayEnv, 4,194,304 games", 19, 4194304, VARIANT_B, AGENT_RANDOM, 30, 6000, dev, peak),   # ~36 episodes: the games must be out of phase, in compressible
            # memory the step time follows how full the boards are (726-891 us over a cohort that is still in step, profiles/r2v)
        ]
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(N, args.cpu_budget)
        print(json.dumps(line), file=args.out, flush=True)
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """Keep stdout for the ONE JSON line: libraries (NCCL prints "NCCL version ..." there when NCCL_DEBUG is set) write to
    file descriptor 1, so point descriptor 1 at stderr and return a private handle to the real stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--board", type=int, default=BOARD)
    ap.add_argument("--games-per-gpu", type=int, default=GAMES_PER_GPU)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=40)
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every step from Python instead of replaying a CUDA graph")
    ap.add_argument("--preroll", type=int, default=2000, help="untimed env steps (one hexb_rollout launch) before warm-up: de-synchronises the games")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_configs block of the 1-GPU line")
    ap.add_argument("--ref-budget", type=float, default=45.0, help="--impl reference: seconds of CPU sampling in total")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's obs / mask / reward / done "
                    "(rank 0's games, a fixed sample of at most 48 MiB) as DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device path's outputs; the reference arm has none")
    args.out = _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
