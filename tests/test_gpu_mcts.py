"""GPU (-m gpu): the batched tree search (hexb_mcts_*) through libhexb.so - whole trees against the oracle (N = 3..19) and the host
emulator (11x11, G = 173, S = 200), sharding, both obs dtypes, torch.ops.hexb against the MCTS class, CUDA graphs of both forms,
one-move wins, and MCTS against flat Monte-Carlo."""
import os
import sys

import numpy as np
import pytest
import torch

from emu import mcts_emu
from emu.emu import EmuBatch
import mcts_common as mc
import search_common as sc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hb():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import hex_gym_env_b200 as hb
    return hb


def host(ex):
    return {k: v.cpu().numpy() for k, v in ex.items()}


def env_batch(hb, N, G, seed, variant, agent_mode, opp_first, steps=None, obs_dtype=torch.int8, game_offset=0):
    env = hb.HexBatch(N, G, variant=variant, device=0, seed=seed, agent_mode=agent_mode, opponent_first=opp_first,
                      obs_dtype=obs_dtype, game_offset=game_offset)
    env.reset()
    for _ in range(sc.env_steps(N) if steps is None else steps):
        env.step(outputs=False)
    return env


def tree_of(t):
    return mc.parse_tree(t.tree.cpu().numpy(), t.batch.N, t.batch.G)


def split_rounds(t, S, rng, orc=None):
    """S select / expand rounds with seeded priors and values; the oracle's trees follow when given."""
    G, C = t.batch.G, t.batch.C
    for _ in range(S):
        obs, mask, pending = t.select()
        obs, mask, pending = obs.cpu().numpy(), mask.cpu().numpy(), pending.cpu().numpy()
        if orc is not None:
            for g, o in enumerate(orc):
                want = o.select() if o is not None else None
                assert pending[g] == (want is not None), g
                if want is not None:
                    assert np.array_equal(obs[g], want[0]) and np.array_equal(mask[g], want[1]), g
        priors = rng.dirichlet(np.ones(C), size=G).astype(np.float32)
        values = rng.uniform(-1, 1, size=G).astype(np.float32)
        t.expand(torch.from_numpy(priors).cuda(), torch.from_numpy(values).cuda())
        if orc is not None:
            for g, o in enumerate(orc):
                if o is not None and pending[g]:
                    o.expand(priors[g], values[g])


@pytest.mark.parametrize("N", range(3, 20))
def test_trees_match_the_oracle(hb, N):
    """Fused and split forms, env handles of every kind and raw handles of both variants, small G and S, a pool that fills."""
    rng = np.random.default_rng(N)
    S = 16 if N <= 9 else 6
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 40 * N + 10 * variant + agent_mode
        env = env_batch(hb, N, 3, seed, variant, agent_mode, opp_first)
        t = hb.MCTS(env, 3 * S, c_puct=1.5, fpu=0.25)
        t.reset(first_playout=5)
        t.search(S, 2)
        orc = mc.oracle_trees(host(env.export_state()), seed, 0, variant, 3 * S, 1.5, 0.25, 5)
        for o in orc:
            for _ in range(S if o is not None else 0):
                o.simulate(2)
        mc.assert_trees_equal(tree_of(t), orc)
    for variant in (0, 1):
        raw = hb.HexBatch(N, 4, variant=variant, device=0, seed=9, game_offset=2, raw=True)
        boards, to_move = sc.random_boards(rng, 4, N)
        raw.import_boards(np.where(rng.uniform(size=boards.shape) < 0.5, 2, boards).astype(np.int8), to_move)
        t = hb.MCTS(raw, S // 2, c_puct=1.1, fpu=-0.2)
        t.reset()
        orc = mc.oracle_trees(host(raw.export_state()), 9, 2, variant, S // 2, 1.1, -0.2, 0)
        split_rounds(t, S, rng, orc)
        mc.assert_trees_equal(tree_of(t), orc)


def emu_env(N, G, seed, variant, agent_mode, opp_first):
    env = EmuBatch(variant, N, G, seed=seed, agent_mode=agent_mode, opponent_first=opp_first)
    env.reset()
    for _ in range(sc.env_steps(N)):
        env.step()
    return env


def test_fused_and_split_match_the_emulator_at_11x11(hb):
    N, G, S, P = 11, 173, 200, 4
    env = env_batch(hb, N, G, 31, 1, 2, False)
    emu = emu_env(N, G, 31, 1, 2, False)
    assert np.array_equal(host(env.export_state())["regions"], emu.export()["regions"])
    t = hb.MCTS(env, 150, c_puct=1.25, fpu=0.5)                       # the pool fills before S + 1
    e = mcts_emu.EmuMCTS(emu, 150, 1.25, 0.5)
    t.reset(first_playout=7)
    e.reset(first_playout=7)
    t.search(S, P)
    e.search(S, P)
    mc.assert_same_tree(t.tree.cpu().numpy(), e.tree, N, G)
    got, want = t.root(), e.root()
    for a, b in zip(got, want):
        assert np.array_equal(a.cpu().numpy(), b)
    t.reset()
    e.reset()
    rng_a, rng_b = np.random.default_rng(1), np.random.default_rng(1)
    split_rounds(t, 60, rng_a)
    for _ in range(60):
        e.select()
        e.expand(rng_b.dirichlet(np.ones(N * N), size=G).astype(np.float32), rng_b.uniform(-1, 1, size=G).astype(np.float32))
    mc.assert_same_tree(t.tree.cpu().numpy(), e.tree, N, G)


def test_sharding_does_not_change_the_search(hb):
    """Two shards (game_offset) of the same positions search what one batch does: playout streams key on the global index."""
    N, G, H = 7, 200, 83
    rng = np.random.default_rng(4)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.5, 2, boards).astype(np.int8)
    out = []
    for off, n in ((0, G), (0, H), (H, G - H)):
        raw = hb.HexBatch(N, n, variant=1, device=0, seed=17, game_offset=off, raw=True)
        raw.import_boards(boards[off:off + n], to_move[off:off + n])
        t = hb.MCTS(raw, 100)
        t.reset()
        t.search(120, 4)
        out.append([x.cpu() for x in t.root()])
    for k in range(4):
        assert torch.equal(out[0][k], torch.cat([out[1][k], out[2][k]])), k


def test_obs_dtypes_agree(hb):
    """select writes the leaf in the handle's obs dtype: float32 leaves are the int8 leaves converted."""
    N, G = 9, 64
    outs = []
    for dt in (torch.int8, torch.float32):
        env = env_batch(hb, N, G, 3, 1, 2, False, obs_dtype=dt)
        t = hb.MCTS(env, 40)
        t.reset()
        rounds = []
        for _ in range(12):
            obs, mask, pending = t.select()
            assert obs.dtype == dt
            rounds.append((obs.float().clone(), mask.clone(), pending.clone()))
            t.expand(torch.full((G, N * N), 0.5, device="cuda"), torch.full((G,), 0.1, device="cuda"))
        outs.append(rounds)
    for (a, b) in zip(*outs):
        p = a[2].bool()
        assert torch.equal(a[2], b[2]) and torch.equal(a[0][p], b[0][p]) and torch.equal(a[1][p], b[1][p])


def test_torch_ops_equal_the_class_and_graphs_equal_eager(hb):
    from hex_gym_env_b200 import torch_ops
    ops = torch_ops.load()
    N, G, S, P = 8, 96, 50, 4
    env = env_batch(hb, N, G, 12, 1, 2, False)
    a, b, c = (hb.MCTS(env, S + 1, c_puct=1.2) for _ in range(3))
    a.reset(first_playout=3)
    a.search(S, P)
    want = a.root()
    ops.mcts_init(env.handle, b.tree, S + 1, 1.2, 0.0, 3, None)
    ops.mcts_search(env.handle, b.tree, S, P)
    got = [torch.empty_like(x) for x in want]
    ops.mcts_root(env.handle, b.tree, *got)
    same = lambda x, y: mc.assert_same_tree(x.cpu().numpy(), y.cpu().numpy(), N, G)
    same(a.tree, b.tree)
    assert all(torch.equal(x, y) for x, y in zip(got, want))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        c.reset()
        s.synchronize()
        with torch.cuda.graph(graph, stream=s):
            ops.mcts_init(env.handle, c.tree, S + 1, 1.2, 0.0, 3, None)
            ops.mcts_search(env.handle, c.tree, S, P)
    torch.cuda.current_stream().wait_stream(s)
    c.tree.zero_()
    graph.replay()
    torch.cuda.synchronize()
    same(c.tree, a.tree)
    # split form: select -> a fixed torch "network" -> expand, eager against a graph of the same rounds
    C = N * N
    w = torch.randn(C, C, generator=torch.Generator().manual_seed(0)).cuda()
    leaf = [torch.zeros(G, N, N, dtype=torch.int8, device="cuda"), torch.zeros(G, C, dtype=torch.uint8, device="cuda"),
            torch.zeros(G, dtype=torch.uint8, device="cuda")]
    pri, val = torch.zeros(G, C, device="cuda"), torch.zeros(G, device="cuda")

    def rounds(tree, n):
        for _ in range(n):
            ops.mcts_select(env.handle, tree, *leaf)
            logits = leaf[0].view(G, C).float() @ w
            pri.copy_(torch.softmax(logits.masked_fill(leaf[1] == 0, -1e9), 1))
            val.copy_(torch.tanh(logits.mean(1)))
            ops.mcts_expand(env.handle, tree, pri, val)

    a.reset()
    rounds(a.tree, 30)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        rounds(c.tree, 1)
        s.synchronize()
        with torch.cuda.graph(graph, stream=s):
            rounds(c.tree, 30)
    torch.cuda.current_stream().wait_stream(s)
    c.reset()
    graph.replay()
    torch.cuda.synchronize()
    same(c.tree, a.tree)
    with pytest.raises(RuntimeError):
        ops.mcts_search(env.handle, c.tree, 0, 1)
    with pytest.raises(RuntimeError):
        ops.mcts_init(env.handle, c.tree[:1024], S + 1, 1.2, 0.0, 0, None)            # smaller than the tree


def test_argument_checks(hb):
    env = hb.HexBatch(5, 8, variant=1, device=0, seed=1, agent_mode=2)
    with pytest.raises(ValueError):
        hb.MCTS(env, 0)
    t = hb.MCTS(env, 10)
    with pytest.raises(RuntimeError):
        t.search(1, 1)                                                                 # before reset
    t.reset()
    with pytest.raises(ValueError):
        t.search(0, 1)
    with pytest.raises(ValueError):
        t.search(1, 0)
    with pytest.raises(ValueError):
        t.expand(torch.zeros(8, 24, device="cuda"), torch.zeros(8, device="cuda"))
    from hex_gym_env_b200 import _native
    L = _native.lib()
    p = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    assert L.hexb_mcts_init(env._h, p.data_ptr(), 64, 10, 1.0, 0.0, 0, None, None) == -3      # HEXB_ERR_STATE: too small
    assert L.hexb_mcts_init(env._h, p.data_ptr(), t.tree_bytes, 0, 1.0, 0.0, 0, None, None) == -1
    assert L.hexb_mcts_search(env._h, p.data_ptr(), t.tree_bytes, 1, 0, None) == -1


# Positions with a winning cell for the side to move (mcts_common.one_move_win_positions, 7x7, seed 2024), S = 100, P = 4,
# c_puct 1, fpu 1: the most visited root cell wins in 230 of 256 positions, computed by the emulator (tests/emu) before any GPU
# run; the device must reproduce the emulator's visits exactly.
ONE_MOVE_WINS = 230


def test_one_move_wins(hb):
    from oracle import mcts
    N, G, S, P = 7, 256, 100, 4
    boards, movers, wins = mc.one_move_win_positions(np.random.default_rng(2024), G, N)
    raw = hb.HexBatch(N, G, variant=1, device=0, seed=11, raw=True)
    raw.import_boards(boards, movers)
    t = hb.MCTS(raw, S + 1, c_puct=1.0, fpu=1.0)
    t.reset()
    t.search(S, P)
    visits = t.root()[0].cpu().numpy()
    emu = EmuBatch(1, N, G, seed=11, raw=True)
    emu.import_boards(boards, movers)
    e = mcts_emu.EmuMCTS(emu, S + 1, 1.0, 1.0)
    e.reset()
    e.search(S, P)
    assert np.array_equal(visits, e.root()[0])
    a = visits.argmax(1)
    cell = np.array([mcts.action(1, int(movers[g]), N, int(a[g])) for g in range(G)])
    hit = int(wins[np.arange(G), cell].sum())
    print("one-move wins: the most visited cell wins in %d of %d positions" % (hit, G))
    assert hit == ONE_MOVE_WINS


# examples/mcts_vs_flat_mc.py at 5x5, 512 games, MCTS 200 simulations x 4 playouts (c_puct 1, fpu 1) against flat MC with 32
# playouts per cell: 800 playouts per move each. Deterministic given the seeds. Measured on a B200: MCTS won 378 of 512 games
# (0.738; 95 % interval 0.699-0.774), 215 of 256 as BLACK and 163 of 256 as WHITE.
MCTS_VS_FLAT_MIN_WIN_RATE = 0.70


def test_mcts_vs_flat_mc_example(hb):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    try:
        import mcts_vs_flat_mc
    finally:
        sys.path.pop(0)
    r = mcts_vs_flat_mc.run(board_size=5, games=512, sims=200, playouts=4, seed=0)
    print("mcts_vs_flat_mc 5x5: MCTS won %d of %d (%.4f, 95%% interval %.4f-%.4f; %d as BLACK, %d as WHITE)"
          % (r["mcts_wins"], r["games"], r["win_rate"], r["interval95"][0], r["interval95"][1], r["mcts_black_wins"],
             r["mcts_white_wins"]))
    assert r["win_rate"] > MCTS_VS_FLAT_MIN_WIN_RATE
