"""GPU (-m gpu): bridge-reply playouts (include/hexb.h, HEXB_PLAYOUT_BRIDGE) through libhexb.so - playouts_policy and whole
search_policy trees against the restated rule (tests/bridge_oracle.py) for N = 3..19 and against the host emulator at 11x11
(G = 173, S = 200), policy 0 of the new entries byte for byte against the old ones, torch.ops.hexb against the class, a CUDA graph
of a bridge search, sharding, and positions where the opponent has just intruded into a bridge of the side to move."""
import numpy as np
import pytest
import torch

import bridge_oracle as bo
import mcts_common as mc
import search_common as sc
from emu.emu import EmuBatch, EmuMCTS, playouts
from oracle import mcts, playout

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hb():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import hex_gym_env_b200 as hb
    return hb


def host(ex):
    return {k: v.cpu().numpy() for k, v in ex.items()}


def env_batch(hb, N, G, seed, variant, agent_mode, opp_first, steps=None, game_offset=0):
    env = hb.HexBatch(N, G, variant=variant, device=0, seed=seed, agent_mode=agent_mode, opponent_first=opp_first,
                      game_offset=game_offset)
    env.reset()
    for _ in range(sc.env_steps(N) if steps is None else steps):
        env.step(outputs=False)
    return env


def tree_of(t):
    return mc.parse_tree(t.tree.cpu().numpy(), t.batch.N, t.batch.G)


def oracle_wins(ex, seed, game_offset, first, P, policy):
    boards = sc.true_boards(ex)
    out = np.full(len(ex["cur"]), -1, np.int32)
    for g in range(len(out)):
        if not ex["done"][g]:
            out[g] = bo.wins(boards[g], int(ex["cur"][g]), seed, game_offset + g, first, P, policy)
    return out


def oracle_trees(ex, seed, game_offset, variant, max_nodes, c_puct, fpu, first):
    boards = sc.true_boards(ex)
    return [bo.RootTree(boards[g], int(ex["cur"][g]), max_nodes, c_puct, fpu, first, variant, seed, game_offset + g)
            if not ex["done"][g] else None for g in range(len(ex["cur"]))]


@pytest.mark.parametrize("N", range(3, 20))
def test_bridge_playouts_match_the_rule(hb, N):
    """Env games of every kind (WHITE agents stored transposed) and raw games of both variants, P = 37, first_playout > 0."""
    rng = np.random.default_rng(N)
    G, P, first = 3, 37, 5
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 1000 * N + 10 * variant + agent_mode
        env = env_batch(hb, N, G, seed, variant, agent_mode, opp_first)
        got = env.playouts(P, first, policy=hb.PLAYOUT_BRIDGE).cpu().numpy()
        assert np.array_equal(got, oracle_wins(host(env.export_state()), seed, 0, first, P, bo.PLAYOUT_BRIDGE)), (variant, agent_mode)
    for variant in (0, 1):
        raw = hb.HexBatch(N, G, variant=variant, device=0, seed=77, game_offset=5, raw=True)
        boards, to_move = sc.random_boards(rng, G, N)
        raw.import_boards(np.where(rng.uniform(size=boards.shape) < 0.5, 2, boards).astype(np.int8), to_move)
        got = raw.playouts(P, first, policy=hb.PLAYOUT_BRIDGE).cpu().numpy()
        assert np.array_equal(got, oracle_wins(host(raw.export_state()), 77, 5, first, P, bo.PLAYOUT_BRIDGE)), variant


@pytest.mark.parametrize("N", range(3, 20))
def test_bridge_trees_match_the_rule(hb, N):
    """Whole trees of search(S, 2, PLAYOUT_BRIDGE): env handles of every kind and raw handles of both variants, a pool that fills."""
    rng = np.random.default_rng(100 + N)
    S = 16 if N <= 9 else 6
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 40 * N + 10 * variant + agent_mode
        env = env_batch(hb, N, 3, seed, variant, agent_mode, opp_first)
        t = hb.MCTS(env, 3 * S, c_puct=1.5, fpu=0.25)
        t.reset(first_playout=5)
        t.search(S, 2, policy=hb.PLAYOUT_BRIDGE)
        orc = oracle_trees(host(env.export_state()), seed, 0, variant, 3 * S, 1.5, 0.25, 5)
        for o in orc:
            for _ in range(S if o is not None else 0):
                o.simulate(2, bo.PLAYOUT_BRIDGE)
        mc.assert_trees_equal(tree_of(t), orc)
    for variant in (0, 1):
        raw = hb.HexBatch(N, 4, variant=variant, device=0, seed=9, game_offset=2, raw=True)
        boards, to_move = sc.random_boards(rng, 4, N)
        raw.import_boards(np.where(rng.uniform(size=boards.shape) < 0.5, 2, boards).astype(np.int8), to_move)
        t = hb.MCTS(raw, S // 2, c_puct=1.1, fpu=-0.2)
        t.reset(first_playout=2 ** 32 - 7)                                   # playout indices wrap mod 2^32
        t.search(S, 3, policy=hb.PLAYOUT_BRIDGE)
        orc = oracle_trees(host(raw.export_state()), 9, 2, variant, S // 2, 1.1, -0.2, 2 ** 32 - 7)
        for o in orc:
            for _ in range(S if o is not None else 0):
                o.simulate(3, bo.PLAYOUT_BRIDGE)
        mc.assert_trees_equal(tree_of(t), orc)


def emu_env(N, G, seed, variant, agent_mode, opp_first):
    env = EmuBatch(variant, N, G, seed=seed, agent_mode=agent_mode, opponent_first=opp_first)
    env.reset()
    for _ in range(sc.env_steps(N)):
        env.step()
    return env


def test_bridge_search_and_playouts_match_the_emulator_at_11x11(hb):
    N, G, S, P = 11, 173, 200, 4
    env = env_batch(hb, N, G, 31, 1, 2, False)
    emu = emu_env(N, G, 31, 1, 2, False)
    assert np.array_equal(host(env.export_state())["regions"], emu.export()["regions"])
    assert np.array_equal(env.playouts(96, 3, policy=hb.PLAYOUT_BRIDGE).cpu().numpy(),
                          playouts(emu, 96, 3, policy=hb.PLAYOUT_BRIDGE))
    t = hb.MCTS(env, 150, c_puct=1.25, fpu=0.5)                            # the pool fills before S + 1
    e = EmuMCTS(emu, 150, 1.25, 0.5)
    t.reset(first_playout=7)
    e.reset(first_playout=7)
    t.search(S, P, policy=hb.PLAYOUT_BRIDGE)
    e.search(S, P, hb.PLAYOUT_BRIDGE)
    mc.assert_same_tree(t.tree.cpu().numpy(), e.tree, N, G)
    for a, b in zip(t.root(), e.root()):
        assert np.array_equal(a.cpu().numpy(), b)


def test_policy_zero_is_the_old_entries_byte_for_byte(hb):
    """hexb_playouts_policy(0) writes what hexb_playouts writes, and hexb_mcts_search_policy(0) leaves the whole tree buffer as
    hexb_mcts_search does (called through the C ABI directly)."""
    import ctypes
    from hex_gym_env_b200 import _native
    L = _native.lib()
    N, G, S, P = 9, 300, 60, 8
    env = env_batch(hb, N, G, 5, 1, 2, False)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    w_old, w_new = (torch.full((G,), -7, dtype=torch.int32, device="cuda") for _ in range(2))
    assert L.hexb_playouts(env._h, 64, 11, None, ctypes.c_void_p(w_old.data_ptr()), stream) == 0
    assert L.hexb_playouts_policy(env._h, 64, 11, 0, None, ctypes.c_void_p(w_new.data_ptr()), stream) == 0
    assert torch.equal(w_old, w_new) and torch.equal(w_new, env.playouts(64, 11))
    a, b = hb.MCTS(env, S + 1), hb.MCTS(env, S + 1)
    for t in (a, b):
        t.tree.fill_(0x5a)                                                 # bytes the search leaves alone compare too
        t.reset(first_playout=4)
    h, ta, nb = a._args()
    _, tb, _ = b._args()
    assert L.hexb_mcts_search(h, ta, nb, S, P, stream) == 0
    assert L.hexb_mcts_search_policy(h, tb, nb, S, P, 0, stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(a.tree, b.tree)
    for bad in (-1, 2):
        assert L.hexb_playouts_policy(env._h, 8, 0, bad, None, ctypes.c_void_p(w_new.data_ptr()), stream) == -1
        assert L.hexb_mcts_search_policy(h, tb, nb, 1, 1, bad, stream) == -1
        with pytest.raises(ValueError):
            env.playouts(8, policy=bad)
        with pytest.raises(ValueError):
            b.search(1, 1, policy=bad)
    torch.cuda.synchronize()
    assert torch.equal(a.tree, b.tree)                                     # a refused call launches nothing


def test_torch_ops_graphs_and_sharding(hb):
    """torch.ops.hexb.playouts / mcts_search with policy=1 equal the class; a captured CUDA graph of a bridge search equals eager;
    two shards (game_offset) search what one batch does."""
    from hex_gym_env_b200 import torch_ops
    ops = torch_ops.load()
    N, G, S, P = 8, 96, 50, 4
    env = env_batch(hb, N, G, 12, 1, 2, False)
    wins = torch.empty(G, dtype=torch.int32, device="cuda")
    ops.playouts(env.handle, 64, 2, None, wins, policy=1)
    assert torch.equal(wins, env.playouts(64, 2, policy=hb.PLAYOUT_BRIDGE))
    ops.playouts(env.handle, 64, 2, None, wins)                           # the default stays random
    assert torch.equal(wins, env.playouts(64, 2))
    a, b, c = (hb.MCTS(env, S + 1, c_puct=1.2) for _ in range(3))
    a.reset(first_playout=3)
    a.search(S, P, policy=hb.PLAYOUT_BRIDGE)
    ops.mcts_init(env.handle, b.tree, S + 1, 1.2, 0.0, 3, None)
    ops.mcts_search(env.handle, b.tree, S, P, policy=1)
    same = lambda x, y: mc.assert_same_tree(x.cpu().numpy(), y.cpu().numpy(), N, G)
    same(a.tree, b.tree)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        c.reset()
        s.synchronize()
        with torch.cuda.graph(graph, stream=s):
            ops.mcts_init(env.handle, c.tree, S + 1, 1.2, 0.0, 3, None)
            ops.mcts_search(env.handle, c.tree, S, P, policy=1)
    torch.cuda.current_stream().wait_stream(s)
    c.tree.zero_()
    graph.replay()
    torch.cuda.synchronize()
    same(c.tree, a.tree)
    with pytest.raises(RuntimeError):
        ops.mcts_search(env.handle, c.tree, S, P, policy=2)
    with pytest.raises(RuntimeError):
        ops.playouts(env.handle, 8, 0, None, wins, policy=-1)
    # sharding
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
        t.search(120, 4, policy=hb.PLAYOUT_BRIDGE)
        out.append([x.cpu() for x in t.root()] + [raw.playouts(40, 1, policy=hb.PLAYOUT_BRIDGE).cpu()])
    for k in range(5):
        assert torch.equal(out[0][k], torch.cat([out[1][k], out[2][k]])), k


# ---------------------------------------------------------------------------------------------- intrusion positions
BRIDGE_STEPS = ((2, -1), (1, 1), (1, -2))   # (dy, dx) from one stone of a bridge to the other, downwards


def intrusion_positions(rng, G, N, noise=0.15):
    """G 7x7-style positions (true boards, side to move, the answer cell): the side to move has a chain of bridges from its edge
    to its other edge (edge bridges at both ends), and the opponent has just played into one carrier; the answer is the other
    carrier cell, after which the chain is a virtual connection. Random stones elsewhere; nobody has connected yet. BLACK
    positions are built directly, WHITE ones as their transposes with the colours swapped."""
    boards, movers, answers = [], [], []
    while len(boards) < G:
        y, x = 1, int(rng.integers(0, N - 1))
        stones, carriers = [(y, x)], [((0, x), (0, x + 1))]
        while y < N - 2:
            dy, dx = BRIDGE_STEPS[int(rng.integers(0, 3))]
            if y + dy > N - 2 or not 0 <= x + dx < N:
                if x + 1 < N and rng.uniform() < 0.5:
                    dy, dx = 1, 1
                else:
                    continue
            carriers.append({(2, -1): ((y + 1, x - 1), (y + 1, x)), (1, 1): ((y, x + 1), (y + 1, x)),
                             (1, -2): ((y, x - 1), (y + 1, x - 1))}[(dy, dx)])
            y, x = y + dy, x + dx
            stones.append((y, x))
        if x < 1:
            continue
        carriers.append(((N - 1, x - 1), (N - 1, x)))
        b = np.where(rng.uniform(size=(N, N)) < noise, rng.integers(0, 2, size=(N, N)), 2).astype(np.int8)
        for pair in carriers:
            for q in pair:
                b[q] = 2
        for q in stones:
            b[q] = 0
        k, j = int(rng.integers(0, len(carriers))), int(rng.integers(0, 2))
        b[carriers[k][j]] = 1
        ans = carriers[k][1 - j]
        if playout.connects(b, 0) or playout.connects(b, 1):
            continue
        t = 0
        if rng.uniform() < 0.5:
            b, t, ans = np.where(b == 2, 2, 1 - b).T.copy(), 1, (ans[1], ans[0])
        boards.append(b)
        movers.append(t)
        answers.append(ans[0] * N + ans[1])
    return np.stack(boards), np.array(movers, np.int8), np.array(answers)


# intrusion_positions(np.random.default_rng(2025), 256, 7), S = 100, P = 4, c_puct 1, fpu 1, seed 13: the most visited root cell
# is the answer in 32 positions with random playouts and in 93 with bridge playouts, computed by the emulator (tests/emu) before
# any GPU run; the device must reproduce the emulator's visits exactly.
INTRUSION_ANSWERS = {0: 32, 1: 93}


def test_bridge_search_answers_intrusions(hb):
    N, G, S, P = 7, 256, 100, 4
    boards, movers, answers = intrusion_positions(np.random.default_rng(2025), G, N)
    hits = {}
    for policy in (hb.PLAYOUT_RANDOM, hb.PLAYOUT_BRIDGE):
        raw = hb.HexBatch(N, G, variant=1, device=0, seed=13, raw=True)
        raw.import_boards(boards, movers)
        t = hb.MCTS(raw, S + 1, c_puct=1.0, fpu=1.0)
        t.reset()
        t.search(S, P, policy=policy)
        visits = t.root()[0].cpu().numpy()
        emu = EmuBatch(1, N, G, seed=13, raw=True)
        emu.import_boards(boards, movers)
        e = EmuMCTS(emu, S + 1, 1.0, 1.0)
        e.reset()
        e.search(S, P, policy)
        assert np.array_equal(visits, e.root()[0]), policy
        a = visits.argmax(1)
        cell = np.array([mcts.action(1, int(movers[g]), N, int(a[g])) for g in range(G)])
        hits[policy] = int((cell == answers).sum())
    print("intrusion answers of %d positions: random playouts %d, bridge playouts %d" % (G, hits[0], hits[1]))
    assert hits == INTRUSION_ANSWERS and hits[1] > hits[0]
