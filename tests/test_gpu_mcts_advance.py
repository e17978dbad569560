"""GPU (-m gpu): tree reuse across moves (hexb_mcts_advance) through libhexb.so - whole trees and root positions against the
restatement of the definition (mcts_advance_common.advance) for N = 3..19 over move chains in both forms and every handle kind, byte-identical
trees against the host emulator at 11x11, torch.ops.hexb.mcts_advance against the MCTS class, a CUDA graph of search -> ply ->
advance against eager, sharding, and the reuse example against the emulator's win count."""
import os
import sys

import numpy as np
import pytest
import torch

from emu import mcts_advance_emu
from emu.emu import EmuBatch
import mcts_advance_common as ma
import mcts_common as mc
import search_common as sc

pytestmark = pytest.mark.gpu

C_PUCT, FPU = 1.3, 0.1


@pytest.fixture(scope="module")
def hb():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import hex_gym_env_b200 as hb
    return hb


def host(ex):
    return {k: v.cpu().numpy() for k, v in ex.items()}


def check(t, orc):
    ma.assert_advanced_trees_equal(t.tree.cpu().numpy(), t.batch.N, t.batch.G, orc)


def grow(t, orc, form, S, rng, P=2):
    """S simulations on the device and on the oracle's trees: fused search, or select / expand with seeded priors and values."""
    if form == "fused":
        t.search(S, P)
        for o in orc:
            for _ in range(S if o is not None else 0):
                o.simulate(P)
        return
    G, C = t.batch.G, t.batch.C
    for _ in range(S):
        obs, mask, pending = (x.cpu().numpy() for x in t.select())
        for g, o in enumerate(orc):
            want = o.select() if o is not None else None
            assert pending[g] == (want is not None), g
            if want is not None:
                assert np.array_equal(obs[g], want[0]) and np.array_equal(mask[g], want[1]), g
        priors = rng.dirichlet(np.ones(C), size=G).astype(np.float32)
        values = rng.uniform(-1, 1, size=G).astype(np.float32)
        t.expand(torch.from_numpy(priors).cuda(), torch.from_numpy(values).cuda())
        for g, o in enumerate(orc):
            if o is not None and pending[g]:
                o.expand(priors[g], values[g])


def most_visited(t, rng, explore=0.2):
    """The root's most visited action per game, a random one for some games (unvisited and illegal ones too)."""
    a = t.root()[0].argmax(1).to(torch.int32).cpu().numpy()
    r = rng.uniform(size=len(a)) < explore
    a[r] = rng.integers(0, t.batch.C, size=int(r.sum()))
    return a


@pytest.mark.parametrize("N", range(3, 20))
def test_chains_match_the_restatement(hb, N):
    """Raw handles of both variants (one ply, then two, alternating) and env handles of every kind (step: the agent's move and
    the opponent's reply, episode ends and auto-resets), both forms, a chain of five moves with an advance after each."""
    rng = np.random.default_rng(N)
    S = 12 if N <= 9 else 4
    kinds = [("raw", v, None) for v in (0, 1)] + [("env", k[0], k) for k in sc.ENV_KINDS]
    for i, (kind, variant, ek) in enumerate(kinds):
        form = ("fused", "split")[i % 2]
        seed = 30 * N + i
        if kind == "raw":
            batch = hb.HexBatch(N, 4, variant=variant, device=0, seed=seed, game_offset=1, raw=True)
            boards, to_move = sc.random_boards(rng, 4, N)
            batch.import_boards(np.where(rng.uniform(size=boards.shape) < 0.8, 2, boards).astype(np.int8), to_move)
            off = 1
        else:
            batch = hb.HexBatch(N, 3, variant=variant, device=0, seed=seed, agent_mode=ek[1], opponent_first=ek[2])
            batch.reset()
            for _ in range(sc.env_steps(N) // 2):
                batch.step(outputs=False)
            off = 0
        M = 3 * S
        t = hb.MCTS(batch, M, c_puct=C_PUCT, fpu=FPU)
        t.reset(first_playout=4)
        orc = mc.oracle_trees(host(batch.export_state()), seed, off, variant, M, C_PUCT, FPU, 4)
        grow(t, orc, form, S, rng)
        for m in range(5):
            a = torch.from_numpy(most_visited(t, rng)).cuda()
            if kind == "raw":
                for _ in range(1 + m % 2):
                    batch.ply(a)
                    a = torch.from_numpy(rng.integers(0, batch.C, size=batch.G).astype(np.int32)).cuda()
            else:
                batch.step(a, outputs=False)
            t.advance(first_playout=100 * m)
            orc = ma.oracle_advance(orc, host(batch.export_state()), seed, off, variant, M, C_PUCT, FPU, 100 * m)
            check(t, orc)
            grow(t, orc, form, S, rng)
            check(t, orc)


def emu_pair(N, G, seed):
    env = EmuBatch(1, N, G, seed=seed, agent_mode=2)
    env.reset()
    for _ in range(sc.env_steps(N)):
        env.step()
    return env


def test_byte_identical_to_the_emulator_at_11x11(hb):
    """G = 173 env roots, 200 simulations per move, four moves (env steps) with an advance after each, then a split-form round."""
    N, G, S, P = 11, 173, 200, 4
    env = hb.HexBatch(N, G, variant=1, device=0, seed=31, agent_mode=2)
    env.reset()
    for _ in range(sc.env_steps(N)):
        env.step(outputs=False)
    emu = emu_pair(N, G, 31)
    t = hb.MCTS(env, 2 * S + 1, c_puct=1.25, fpu=0.0)
    e = mcts_advance_emu.EmuMCTS(emu, 2 * S + 1, 1.25, 0.0)
    t.reset(first_playout=7)
    e.reset(first_playout=7)
    kept = 0
    for m in range(4):
        t.search(S, P)
        e.search(S, P)
        mc.assert_same_tree(t.tree.cpu().numpy(), e.tree, N, G)
        a = t.root()[0].argmax(1).to(torch.int32)
        assert np.array_equal(a.cpu().numpy(), e.root()[0].argmax(1))
        env.step(a, outputs=False)
        emu.step(a.cpu().numpy())
        t.advance(first_playout=1000 * (m + 1))
        e.advance(first_playout=1000 * (m + 1))
        mc.assert_same_tree(t.tree.cpu().numpy(), e.tree, N, G)
        for x, y in zip(t.root(), e.root()):
            assert np.array_equal(x.cpu().numpy(), y)
        kept += int((t.root()[3] > 1).sum())
    assert kept > 0
    rng_a, rng_b = np.random.default_rng(1), np.random.default_rng(1)
    for _ in range(20):
        t.select()
        e.select()
        t.expand(torch.from_numpy(rng_a.dirichlet(np.ones(N * N), size=G).astype(np.float32)).cuda(),
                 torch.from_numpy(rng_a.uniform(-1, 1, size=G).astype(np.float32)).cuda())
        e.expand(rng_b.dirichlet(np.ones(N * N), size=G).astype(np.float32), rng_b.uniform(-1, 1, size=G).astype(np.float32))
    mc.assert_same_tree(t.tree.cpu().numpy(), e.tree, N, G)


def test_torch_op_and_a_cuda_graph(hb):
    """torch.ops.hexb.mcts_advance equals MCTS.advance; a CUDA graph of search -> ply -> advance, replayed, equals eager."""
    from hex_gym_env_b200 import torch_ops
    ops = torch_ops.load()
    N, G, S, P = 7, 96, 60, 2
    rng = np.random.default_rng(2)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.7, 2, boards).astype(np.int8)
    mask = torch.from_numpy((np.arange(G) % 7 != 3).astype(np.uint8)).cuda()

    def fresh_batch():
        raw = hb.HexBatch(N, G, variant=1, device=0, seed=5, raw=True)
        raw.import_boards(boards, to_move)
        return raw

    ra, rb = fresh_batch(), fresh_batch()
    a, b = hb.MCTS(ra, 2 * S + 1), hb.MCTS(rb, 2 * S + 1)
    for t, r in ((a, ra), (b, rb)):
        t.reset()
        t.search(S, P)
        r.ply(t.root()[0].argmax(1).to(torch.int32))
    a.advance(root_mask=mask, first_playout=9)
    ops.mcts_advance(rb.handle, b.tree, 9, mask)
    mc.assert_same_tree(a.tree.cpu().numpy(), b.tree.cpu().numpy(), N, G)
    assert all(torch.equal(x, y) for x, y in zip(a.root(), b.root()))
    with pytest.raises(RuntimeError):
        ops.mcts_advance(rb.handle, b.tree, -1, None)

    # eager: three rounds of search -> ply -> advance; the graph holds the same three rounds
    act = torch.zeros(G, dtype=torch.int32, device="cuda")

    def rounds(t, r, n):
        for i in range(n):
            t.search(S, P)
            v = t.root()[0]
            act.copy_(v.argmax(1).to(torch.int32))
            r.ply(act)
            t.advance(first_playout=i * 1000)

    re_, rg = fresh_batch(), fresh_batch()
    e, g = hb.MCTS(re_, 2 * S + 1), hb.MCTS(rg, 2 * S + 1)
    e.reset()
    rounds(e, re_, 3)
    g.reset()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        scratch = fresh_batch()
        w = hb.MCTS(scratch, 2 * S + 1)
        w.reset()
        rounds(w, scratch, 1)                                         # load the modules and the batch's buffers on this stream
        rg.ply(torch.full((G,), -1, dtype=torch.int32, device="cuda"))  # no change: -1 is out of range
        g.root()
        s.synchronize()
        with torch.cuda.graph(graph, stream=s):
            rounds(g, rg, 3)
    torch.cuda.current_stream().wait_stream(s)
    rg.import_boards(boards, to_move)                                 # the capture ran nothing: start from the same positions
    g.reset()
    graph.replay()
    torch.cuda.synchronize()
    mc.assert_same_tree(g.tree.cpu().numpy(), e.tree.cpu().numpy(), N, G)
    assert torch.equal(rg.export_state()["regions"], re_.export_state()["regions"])


def test_sharding_does_not_change_the_advance(hb):
    N, G, H = 7, 120, 47
    rng = np.random.default_rng(4)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.6, 2, boards).astype(np.int8)
    out = []
    for off, n in ((0, G), (0, H), (H, G - H)):
        raw = hb.HexBatch(N, n, variant=1, device=0, seed=17, game_offset=off, raw=True)
        raw.import_boards(boards[off:off + n], to_move[off:off + n])
        t = hb.MCTS(raw, 121)
        t.reset()
        for m in range(3):
            t.search(60, 2)
            raw.ply(t.root()[0].argmax(1).to(torch.int32))
            t.advance(first_playout=500 * m)
        t.search(20, 2)
        out.append([x.cpu() for x in t.root()])
    for k in range(4):
        assert torch.equal(out[0][k], torch.cat([out[1][k], out[2][k]])), k


# examples/mcts_reuse.py at 5x5, 64 games, 40 simulations x 2 playouts per move, c_puct 1.25, fpu 0, seed 0: computed by the
# host emulator (tests/emu) before any GPU run - reuse won 36 of 64 games (17 as BLACK, 19 as WHITE). The device must reproduce it.
REUSE_WINS_5X5 = (36, 17, 19)


def test_reuse_example_matches_the_emulator(hb):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    try:
        import mcts_reuse
    finally:
        sys.path.pop(0)
    r = mcts_reuse.run(board_size=5, games=64, sims=40, playouts=2, c_puct=1.25, fpu=0.0, seed=0)
    print("mcts_reuse 5x5: reuse won %d of %d (%d as BLACK, %d as WHITE); an advanced root held %.2f visits"
          % (r["reuse_wins"], r["games"], r["reuse_black_wins"], r["reuse_white_wins"], r["mean_visits_kept"]))
    assert (r["reuse_wins"], r["reuse_black_wins"], r["reuse_white_wins"]) == REUSE_WINS_5X5
    emu = EmuBatch(1, 5, 64, seed=0, raw=True)
    emu.reset()
    w, colour, held = mcts_reuse.play(emu, lambda: mcts_advance_emu.EmuMCTS(emu, 81, 1.25, 0.0), 40, 2, lambda x: x, lambda x: x)
    assert mcts_reuse.summary(w, colour, held, 40, 2)["mean_visits_kept"] == r["mean_visits_kept"]
