"""GPU (-m gpu): the tree search where only the device runs its lane-parallel code - the shuffle argmax, cells and path entries
owned as lane + 32k, the playout split over lanes and its sum, advance's ballot renumbering - checked byte for byte against the
host emulator (one lane, the same source) and the oracle: every board size with P playouts from 1 to 65536 and ragged batches,
lines deeper than 32 and 64 plies, float edges (NaN, signed zeros, infinities, overflow), a playout key past 2^32, and a tree
buffer past 4 GiB."""
import numpy as np
import pytest
import torch

from emu.emu import EmuBatch, EmuMCTS
import mcts_advance_common as ma
import mcts_common as mc
import search_common as sc

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]   # the oracle's float32 edges warn


@pytest.fixture(scope="module")
def hb():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import hex_gym_env_b200 as hb
    return hb


def cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def raw_pair(hb, N, G, variant, seed, rng, game_offset=0, fill=0.5):
    """A raw device batch and a raw emulator batch holding the same random positions."""
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < fill, 2, boards).astype(np.int8)
    dev = hb.HexBatch(N, G, variant=variant, device=0, seed=seed, game_offset=game_offset, raw=True)
    emu = EmuBatch(variant, N, G, seed=seed, game_offset=game_offset, raw=True)
    dev.import_boards(boards, to_move)
    emu.import_boards(boards, to_move)
    return dev, emu


def env_pair(hb, N, G, seed, variant, agent_mode, opp_first):
    """An env device batch and its emulator twin after the same env steps (games at every stage)."""
    dev = hb.HexBatch(N, G, variant=variant, device=0, seed=seed, agent_mode=agent_mode, opponent_first=opp_first)
    emu = EmuBatch(variant, N, G, seed=seed, agent_mode=agent_mode, opponent_first=opp_first)
    dev.reset()
    emu.reset()
    for _ in range(sc.env_steps(N)):
        dev.step(outputs=False)
        emu.step()
    assert np.array_equal(dev.export_state()["regions"].cpu().numpy(), emu.export()["regions"])
    return dev, emu


def same(t, e):
    """Device and emulator trees byte for byte (same_bits for NaNs), and the root() outputs."""
    N, G = t.batch.N, t.batch.G
    mc.assert_same_tree(t.tree.cpu().numpy(), e.tree, N, G)
    mc.assert_root_outputs_equal([x.cpu().numpy() for x in t.root()], e.root())


def split_both(t, e, S, inputs, orc=None):
    """S select / expand rounds on the device, the emulator and (when given) the oracle's trees; select's outputs compared every
    round. inputs(leaf_mask) -> (priors, values)."""
    for _ in range(S):
        obs, mask, pending = (x.cpu().numpy() for x in t.select())
        eo, em, ep = e.select()
        assert np.array_equal(pending, ep)
        rows = ep == 1
        assert np.array_equal(obs[rows], eo[rows]) and np.array_equal(mask[rows], em[rows])
        if orc is not None:
            for g, o in enumerate(orc):
                want = o.select() if o is not None else None
                assert ep[g] == (want is not None), g
                if want is not None:
                    assert np.array_equal(eo[g], want[0]) and np.array_equal(em[g], want[1]), g
        priors, values = inputs(em)
        t.expand(cuda(priors), cuda(values))
        e.expand(priors, values)
        if orc is not None:
            for g, o in enumerate(orc):
                if o is not None and ep[g]:
                    o.expand(priors[g], values[g])


def dirichlet(rng, G, C):
    return lambda mask: (rng.dirichlet(np.ones(C), size=G).astype(np.float32), rng.uniform(-1, 1, size=G).astype(np.float32))


# ---------------------------------------------------------------------------------------------- a. every board size
PLAYOUTS = (1, 31, 32, 33, 100)   # lanes with no playout, one, or several; rotated over N


@pytest.mark.parametrize("N", range(3, 20))
def test_device_equals_the_emulator(hb, N):
    """Env handles of every kind and raw handles of both variants, G not a multiple of 4 (roots per 128-thread block), a pool that
    fills (max_nodes < S + 1): fused search, split search with Dirichlet priors, then a ply (raw) or an env step, advance and more
    fused search."""
    P = PLAYOUTS[N % 5]
    S = 24 if N <= 9 else 12
    G = 9 + 2 * (N % 3) + (N % 2)
    M = 2 * S // 3
    rng = np.random.default_rng(100 + N)
    kinds = [("env", k) for k in sc.ENV_KINDS] + [("raw", v) for v in (0, 1)]
    for i, (kind, k) in enumerate(kinds):
        seed = 20 * N + i
        if kind == "env":
            dev, emu = env_pair(hb, N, G, seed, *k)
        else:
            dev, emu = raw_pair(hb, N, G, k, seed, rng)
        t = hb.MCTS(dev, M, c_puct=1.25, fpu=0.1)
        e = EmuMCTS(emu, M, 1.25, 0.1)
        t.reset(first_playout=3 * N)
        e.reset(first_playout=3 * N)
        t.search(S, P)
        e.search(S, P)
        same(t, e)
        assert (t.root()[3].cpu().numpy() == M).any()
        t.reset()
        e.reset()
        split_both(t, e, S, dirichlet(rng, G, N * N))
        same(t, e)
        a = t.root()[0].argmax(1).to(torch.int32)
        if kind == "env":
            dev.step(a, outputs=False)
            emu.step(a.cpu().numpy())
        else:
            dev.ply(a)
            emu.ply(a.cpu().numpy())
        t.advance(first_playout=1000 + N)
        e.advance(first_playout=1000 + N)
        same(t, e)
        t.search(S // 2, P)
        e.search(S // 2, P)
        same(t, e)
    if N == 3:                                                        # the most playouts per leaf the ABI takes
        dev, emu = raw_pair(hb, N, 3, 1, 7, rng, fill=0.9)
        t, e = hb.MCTS(dev, 4, c_puct=1.25, fpu=0.1), EmuMCTS(emu, 4, 1.25, 0.1)
        t.reset()
        e.reset()
        t.search(3, 65536)
        e.search(3, 65536)
        same(t, e)


# ---------------------------------------------------------------------------------------------- b. deep lines
def depths(roots):
    """The deepest node of each parsed root (through child pointers)."""
    out = []
    for r in roots:
        d = {0: 0}
        for k, nd in enumerate(r["nodes"]):
            if nd["flag"] == 1 and k in d:
                for j in nd["child"][nd["child"] >= 0]:
                    d[int(j)] = d[k] + 1
        out.append(max(d.values()) if r["active"] else 0)
    return out


@pytest.mark.parametrize("N, S, deep, oracle", ((7, 45, 33, True), (9, 50, 33, True), (13, 70, 65, False), (19, 90, 65, False)))
def test_deep_lines(hb, N, S, deep, oracle):
    """Split form with each leaf's prior on one of its legal cells (0 elsewhere) and fpu = -1: every simulation goes one ply
    deeper, so path entries wrap the 32 lanes once (depth > 32) or twice (depth > 64) and mc_backup takes its d += 32 stride. Then
    advance along the line (the kept subtree is a long chain) and go deeper."""
    G = 6
    rng = np.random.default_rng(N)
    dev = hb.HexBatch(N, G, variant=1, device=0, seed=4, raw=True)
    emu = EmuBatch(1, N, G, seed=4, raw=True)
    empty, to_move = np.full((G, N, N), 2, np.int8), (np.arange(G) % 2).astype(np.int8)
    dev.import_boards(empty, to_move)
    emu.import_boards(empty, to_move)
    M = 2 * S + 2
    t, e = hb.MCTS(dev, M, c_puct=1.0, fpu=-1.0), EmuMCTS(emu, M, 1.0, -1.0)
    t.reset()
    e.reset()
    orc = mc.oracle_trees(emu.export(), 4, 0, 1, M, 1.0, -1.0, 0) if oracle else None

    def peaked(mask):
        pri = np.zeros(mask.shape, np.float32)
        for g in range(G):
            legal = np.flatnonzero(mask[g])
            if len(legal):
                pri[g, rng.choice(legal)] = 1.0
        return pri, rng.uniform(-0.5, 0.5, size=G).astype(np.float32)

    for _ in range(S // 10):
        split_both(t, e, 10, peaked, orc)
        same(t, e)
        if orc is not None:
            mc.assert_trees_equal(mc.parse_tree(t.tree.cpu().numpy(), N, G), orc)
    reached = depths(mc.parse_tree(t.tree.cpu().numpy(), N, G))
    assert max(reached) >= deep, reached
    # advance two plies down the line, one at a time: the kept subtree is the rest of the chain
    for _ in range(2):
        a = t.root()[0].argmax(1).to(torch.int32)
        dev.ply(a)
        emu.ply(a.cpu().numpy())
        t.advance()
        e.advance()
        same(t, e)
        if orc is not None:
            orc = ma.oracle_advance(orc, emu.export(), 4, 0, 1, M, 1.0, -1.0, 0)
            ma.assert_advanced_trees_equal(t.tree.cpu().numpy(), N, G, orc)
    kept = depths(mc.parse_tree(t.tree.cpu().numpy(), N, G))
    assert max(kept) >= deep - 2, kept
    split_both(t, e, 10, peaked, orc)
    same(t, e)
    if orc is not None:
        mc.assert_trees_equal(mc.parse_tree(t.tree.cpu().numpy(), N, G), orc)


# ---------------------------------------------------------------------------------------------- c. float edges
@pytest.mark.parametrize("c_puct, fpu", mc.EDGE_SETTINGS)
def test_float_edges(hb, c_puct, fpu):
    """Split form with priors and values from mcts_common.EDGE_PRIORS / EDGE_VALUES (zeros of both signs, subnormals, 3e38, inf,
    NaN) against the emulator and the oracle. A NaN Q + U must rank below every number on the device too, where a NaN has other
    bits than on the host."""
    rng = np.random.default_rng(50 + mc.EDGE_SETTINGS.index((c_puct, fpu)))
    for variant, N in ((0, 4), (1, 5)):
        dev, emu = raw_pair(hb, N, 7, variant, 11, rng)
        t, e = hb.MCTS(dev, 24, c_puct=c_puct, fpu=fpu), EmuMCTS(emu, 24, c_puct, fpu)
        t.reset()
        e.reset()
        orc = mc.oracle_trees(emu.export(), 11, 0, variant, 24, c_puct, fpu, 0)
        split_both(t, e, 30, lambda mask: mc.edge_inputs(rng, 7, N * N), orc)
        same(t, e)
        mc.assert_trees_equal(mc.parse_tree(t.tree.cpu().numpy(), N, 7), orc)


@pytest.mark.parametrize("nan", (0x7fc00000, 0xffc00000, 0x7fffffff))
def test_a_nan_child_gets_no_more_visits(hb, nan):
    """A NaN value backed up through the lowest root edge: that edge gets no further visit while other cells score numbers."""
    N, G = 5, 3
    dev = hb.HexBatch(N, G, variant=1, device=0, seed=3, raw=True)
    emu = EmuBatch(1, N, G, seed=3, raw=True)
    board, to_move = np.full((G, N, N), 2, np.int8), np.zeros(G, np.int8)
    dev.import_boards(board, to_move)
    emu.import_boards(board, to_move)
    t, e = hb.MCTS(dev, 64, c_puct=1.0, fpu=0.0), EmuMCTS(emu, 64, 1.0, 0.0)
    t.reset()
    e.reset()
    orc = mc.oracle_trees(emu.export(), 3, 0, 1, 64, 1.0, 0.0, 0)
    rnd = [0]

    def inputs(mask):
        rnd[0] += 1
        value = np.full(G, 0.5, np.float32)
        if rnd[0] == 2:                                               # round 2's leaf: the child at cell 0
            value[:] = np.array([nan], np.uint32).view(np.float32)[0]
        return np.full((G, N * N), 1.0 / (N * N), np.float32), value

    split_both(t, e, 40, inputs, orc)
    same(t, e)
    mc.assert_trees_equal(mc.parse_tree(t.tree.cpu().numpy(), N, G), orc)
    visits, q = t.root()[0].cpu().numpy(), t.root()[1].cpu().numpy()
    assert np.isnan(q[:, 0]).all() and (visits[:, 0] == 1).all()
    assert ((visits[:, 1:] > 0).sum(1) >= 20).all()


# ---------------------------------------------------------------------------------------------- d. the playout key
@pytest.mark.parametrize("N", (3, 5, 7, 11, 19))
def test_playout_key_past_2_to_the_32(hb, N):
    """game_offset = 12345678901 and first_playout = 2^32 - 40 with P = 33: the playout index wraps mod 2^32 part-way through a
    warp's playouts (lane 0 runs two of them). Against the emulator, and the oracle at N <= 7."""
    off, first, P, S = 12345678901, 2 ** 32 - 40, 33, 8
    rng = np.random.default_rng(N)
    for variant in (0, 1):
        dev, emu = raw_pair(hb, N, 5, variant, 5, rng, game_offset=off)
        t, e = hb.MCTS(dev, S + 1), EmuMCTS(emu, S + 1, 1.25, 0.0)
        t.reset(first_playout=first)
        e.reset(first_playout=first)
        t.search(S, P)
        e.search(S, P)
        same(t, e)
        if N <= 7:
            orc = mc.oracle_trees(emu.export(), 5, off, variant, S + 1, 1.25, 0.0, first)
            for o in orc:
                for _ in range(S if o is not None else 0):
                    o.simulate(P)
            mc.assert_trees_equal(mc.parse_tree(t.tree.cpu().numpy(), N, 5), orc)


# ---------------------------------------------------------------------------------------------- e. a tree past 4 GiB
def test_tree_past_4_gib(hb):
    """19x19, max_nodes 801, G = 1024: 4,931,328 bytes per root, about 5 GB. Roots from g = 871 on start past 2^32 (root 870
    straddles it). A short fused search; the roots around 2^32 and the last ones are checked against an emulator batch of the same
    positions with game_offset = their first index (the playout streams key on the global index), copying only their bytes."""
    N, G, M, S, P = 19, 1024, 801, 16, 2
    rng = np.random.default_rng(19)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.5, 2, boards).astype(np.int8)
    dev = hb.HexBatch(N, G, variant=1, device=0, seed=8, raw=True)
    dev.import_boards(boards, to_move)
    t = hb.MCTS(dev, M)
    t.reset(first_playout=11)
    head = t.tree[:128].cpu().numpy()
    rb = int(head[40:48].view(np.int64)[0])
    assert rb == 4931328 and 128 + 871 * rb >= 2 ** 32 > 128 + 870 * rb and t.tree_bytes > 5 * 10 ** 9
    t.search(S, P)
    visits, q, value, used = (x.cpu().numpy() for x in t.root())
    for lo, hi in ((866, 876), (G - 8, G)):
        n = hi - lo
        emu = EmuBatch(1, N, n, seed=8, game_offset=lo, raw=True)
        emu.import_boards(boards[lo:hi], to_move[lo:hi])
        e = EmuMCTS(emu, M, 1.25, 0.0)
        e.reset(first_playout=11)
        e.search(S, P)
        part = np.concatenate([head, t.tree[128 + lo * rb:128 + hi * rb].cpu().numpy()])
        part[8:16] = np.array([n], np.int64).view(np.uint8)            # the header of an n-root buffer
        mc.assert_same_tree(part, e.tree, N, n)
        mc.assert_root_outputs_equal((visits[lo:hi], q[lo:hi], value[lo:hi], used[lo:hi]), e.root())
        assert (used[lo:hi] > 1).all()
