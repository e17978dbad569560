"""CPU: tree reuse across moves (hexb_mcts_advance) without a GPU - the restatement of the definition (mcts_advance_common.advance) on its
own, and the device code (csrc/hexb_mcts.cuh, mc_advance_root) run by the host emulator against it bit for bit over the whole tree
and the root's position, through chains of moves continued with both search forms, and the argument checks of the C ABI."""
import copy
import ctypes

import numpy as np
import pytest

from emu import mcts_advance_emu
from emu.emu import EmuBatch
from oracle import mcts
from hex_gym_env_b200 import _native
import mcts_advance_common as ma
import mcts_common as mc
import search_common as sc

C_PUCT, FPU = 1.3, 0.1


def raw_batch(N, G, seed, variant, rng, fill=0.6, game_offset=0):
    raw = EmuBatch(variant, N, G, seed=seed, game_offset=game_offset, raw=True)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < fill, 2, boards).astype(np.int8)
    raw.import_boards(boards, to_move)
    return raw


class Pair(object):
    """An emulated tree and the oracle's trees of the same batch, moved on together."""

    def __init__(self, batch, seed, variant, max_nodes, first=1, root_mask=None, game_offset=0, live=None):
        self.batch, self.seed, self.variant, self.max_nodes, self.off = batch, seed, variant, max_nodes, game_offset
        self.e = mcts_advance_emu.EmuMCTS(batch, max_nodes, C_PUCT, FPU)
        self.e.reset(root_mask, first)
        om = root_mask if live is None else (live if root_mask is None else root_mask & live)
        self.orc = mc.oracle_trees(batch.export(), seed, game_offset, variant, max_nodes, C_PUCT, FPU, first, om)
        self.live = live

    def search(self, S, P=2):
        self.e.search(S, P)
        for o in self.orc:
            for _ in range(S if o is not None else 0):
                o.simulate(P)

    def split(self, S, rng):
        G, C = self.batch.G, self.batch.C
        for _ in range(S):
            obs, mask, pending = self.e.select()
            for g, o in enumerate(self.orc):
                want = o.select() if o is not None else None
                assert pending[g] == (want is not None), g
                if want is not None:
                    assert np.array_equal(obs[g], want[0]) and np.array_equal(mask[g], want[1]), g
            priors = rng.dirichlet(np.ones(C), size=G).astype(np.float32)
            values = rng.uniform(-1, 1, size=G).astype(np.float32)
            self.e.expand(priors, values)
            for g, o in enumerate(self.orc):
                if o is not None and pending[g]:
                    o.expand(priors[g], values[g])

    def advance(self, first, root_mask=None):
        self.e.advance(root_mask, first)
        self.orc = ma.oracle_advance(self.orc, self.batch.export(), self.seed, self.off, self.variant, self.max_nodes, C_PUCT, FPU,
                                     first, root_mask, self.live)
        self.check()

    def check(self):
        ma.assert_advanced_trees_equal(self.e.tree, self.batch.N, self.batch.G, self.orc)


def node_at(o, path):
    """The oracle node a path of cells from the root reaches (None: not stored)."""
    k = 0
    for c in path:
        if o.nodes[k].flag != mcts.EXPANDED:
            return None
        k = int(o.nodes[k].child[c])
        if k < 0:
            return None
    return o.nodes[k]


def pick_cells(pair, rng, plies, explore=0.25):
    """plies moves per game, in true cells: the most visited edge of the node the moves so far reach, or (with probability
    explore, or off the tree) a random empty cell. None for a finished game."""
    ex = pair.batch.export()
    boards = sc.true_boards(ex).reshape(pair.batch.G, -1)
    out = []
    for g in range(pair.batch.G):
        if ex["done"][g]:
            out.append(None)
            continue
        b, o, path = boards[g].copy(), pair.orc[g], []
        for _ in range(plies):
            empty = np.flatnonzero(b == 2)
            if len(empty) == 0:
                break
            nd = node_at(o, path) if o is not None else None
            if nd is not None and nd.flag == mcts.EXPANDED and nd.n[empty].max() > 0 and rng.uniform() >= explore:
                c = int(empty[np.argmax(nd.n[empty])])
            else:
                c = int(rng.choice(empty))
            b[c] = 0
            path.append(c)
        out.append(path)
    return out


def ply_paths(pair, paths):
    """Play the paths on a raw batch, one ply per round (games with shorter paths are left alone)."""
    ex = pair.batch.export()
    N, G = pair.batch.N, pair.batch.G
    cur = ex["cur"].astype(int)
    for d in range(max([len(p) for p in paths if p] + [0])):
        acts = np.full(G, -1, np.int32)
        for g, p in enumerate(paths):
            if p and d < len(p):
                acts[g] = mcts.action(pair.variant, cur[g] ^ (d & 1), N, p[d])
        pair.batch.ply(acts)


def env_actions(pair, rng, explore=0.25):
    """Agent actions for an env batch: the root's most visited action, or a random one for some games (illegal ones too)."""
    visits = pair.e.root()[0]
    a = visits.argmax(1).astype(np.int32)
    r = rng.uniform(size=len(a)) < explore
    a[r] = rng.integers(0, pair.batch.C, size=int(r.sum()))
    return a


# ---------------------------------------------------------------------------------------------- the restatement on its own
@pytest.mark.parametrize("N", (4, 5))
def test_oracle_keeps_the_subtree_under_the_played_move(N):
    """After a one-move advance the tree is the old subtree under r node for node (children renumbered), the root's visits are
    the old edge's N and its value is -q of the old root at the played cell, bit for bit."""
    rng = np.random.default_rng(N)
    pair = Pair(raw_batch(N, 6, 5, 1, rng), 5, 1, 400)
    pair.search(120)
    for o in pair.orc:
        if o is None:
            continue
        old = copy.deepcopy(o)
        visits, q, _ = old.root()
        a = int(np.argmax(visits))
        c = mcts.action(1, old.t0, N, a)                  # the root's action convention back to the true cell (an involution)
        r = int(old.nodes[0].child[c])
        board = old.board.copy()
        board[c] = old.t0
        new = ma.advance(o, board, old.t0 ^ 1, 9)
        assert new is o
        keep = ma.reachable(old, r)
        assert len(new.nodes) == len(keep) and keep[0] == r
        ren = {k: i for i, k in enumerate(keep)}
        for i, k in enumerate(keep):
            a_, b_ = new.nodes[i], old.nodes[k]
            assert a_.flag == b_.flag and (i == 0 or a_.nn == b_.nn)
            if b_.flag == mcts.EXPANDED:
                assert np.array_equal(a_.child, [ren[j] if j >= 0 else -1 for j in b_.child])
                assert np.array_equal(a_.n, b_.n) and np.array_equal(a_.w.view(np.uint32), b_.w.view(np.uint32))
                assert np.array_equal(a_.p.view(np.uint32), b_.p.view(np.uint32))
        assert new.s == new.nodes[0].nn == int(old.nodes[0].n[c])
        value = new.root()[2]
        assert np.float32(value).view(np.uint32) == (-q[a]).view(np.uint32)
        assert new.first == 9 and new.t0 == old.t0 ^ 1


def test_root_counters_follow_the_edge_after_a_freed_pool():
    """A node stored only after an advance freed a full pool has Nn below the N of its edge; re-rooting on it takes both root
    counters from the edge. The emulator agrees bit for bit at every stage."""
    N, G = 4, 24
    rng = np.random.default_rng(11)
    pair = Pair(raw_batch(N, G, 3, 0, rng, fill=0.9), 3, 0, 6)
    pair.search(40)
    ply_paths(pair, pick_cells(pair, rng, 1, explore=0.0))
    pair.advance(100)
    pair.search(40)
    pair.check()
    found, paths = 0, []
    for o in pair.orc:
        path = None
        if o is not None and o.nodes[0].flag == mcts.EXPANDED:
            for c in np.flatnonzero(o.nodes[0].child >= 0):
                j = int(o.nodes[0].child[c])
                if o.nodes[j].flag == mcts.EXPANDED and o.nodes[j].nn != o.nodes[0].n[c]:
                    path = [int(c)]
                    found += 1
                    break
        paths.append(path)
    assert found > 0
    edge = [(int(o.nodes[0].n[p[0]]), o.nodes[0].w[p[0]], o.nodes[int(o.nodes[0].child[p[0]])].nn) if p else None
            for o, p in zip(pair.orc, paths)]
    ply_paths(pair, paths)
    pair.advance(200)
    for o, e in zip(pair.orc, edge):
        if e is not None:
            assert o.s == o.nodes[0].nn == e[0] != e[2]
            assert np.float32(o.vsum).view(np.uint32) == (-e[1]).view(np.uint32)


# ---------------------------------------------------------------------------------------------- emulator == restatement
@pytest.mark.parametrize("N", (3, 4, 5, 7, 9, 13))
def test_raw_chains_match(N):
    """Raw handles of both variants, advanced by one ply and by two, over chains of moves; search and select / expand after
    each advance; the pool fills up on the small boards."""
    rng = np.random.default_rng(100 + N)
    S = 24 if N <= 7 else 10
    moves = 6 if N <= 9 else 5
    for variant in (0, 1):
        for form in ("fused", "split"):
            seed = 7 * N + variant
            pair = Pair(raw_batch(N, 5, seed, variant, rng, fill=0.8, game_offset=3), seed, variant, 2 * S, first=2, game_offset=3)
            pair.search(S) if form == "fused" else pair.split(S, rng)
            for m in range(moves):
                ply_paths(pair, pick_cells(pair, rng, 1 + (m % 2)))
                pair.advance(50 * (m + 1))
                pair.search(S) if form == "fused" else pair.split(S, rng)
                pair.check()


@pytest.mark.parametrize("N", (3, 4, 5, 7, 9, 13))
def test_env_chains_match(N):
    """Env handles of every kind advanced by step() (the agent's move and the opponent's reply), episode ends and auto-resets
    included, continued with both forms."""
    rng = np.random.default_rng(200 + N)
    S = 16 if N <= 7 else 8
    moves = 6 if N <= 9 else 5
    for i, (variant, agent_mode, opp_first) in enumerate(sc.ENV_KINDS):
        seed = 11 * N + i
        env = EmuBatch(variant, N, 5, seed=seed, agent_mode=agent_mode, opponent_first=opp_first)
        env.reset()
        for _ in range(sc.env_steps(N) // 2):
            env.step()
        pair = Pair(env, seed, variant, 3 * S)
        form = ("fused", "split")[i % 2]
        pair.search(S) if form == "fused" else pair.split(S, rng)
        for m in range(moves):
            env.step(env_actions(pair, rng))
            pair.advance(m + 1)
            pair.search(S) if form == "fused" else pair.split(S, rng)
            pair.check()


def test_fresh_trees_and_the_kept_tree():
    """k = 0 keeps the tree as it is; three plies, a board with a stone removed, an unvisited move and a move whose child the
    full pool never stored start fresh trees; masked roots become inactive and roots inactive before become fresh ones."""
    N, G = 5, 12
    rng = np.random.default_rng(3)
    raw = raw_batch(N, G, 4, 1, rng, fill=0.9)
    mask = np.ones(G, np.uint8)
    mask[10:] = 0                                                                       # inactive before the advance
    pair = Pair(raw, 4, 1, 40, root_mask=mask)
    pair.search(60)
    before = mc.parse_tree(pair.e.tree, N, G)
    pair.advance(7)                                                                     # k = 0 everywhere
    after = mc.parse_tree(pair.e.tree, N, G)
    mc.assert_trees_equal(after[:10], [mc.as_oracle(r) for r in before[:10]])
    assert all(r["active"] and r["used"] == 1 and r["s"] == 0 for r in after[10:])       # fresh trees
    assert int(pair.e.tree[32:40].view(np.int64)[0]) == 7
    ex = raw.export()
    boards = sc.true_boards(ex).reshape(G, -1)
    paths = pick_cells(pair, rng, 1, explore=0.0)
    kinds = {}
    for g in range(G):
        o = pair.orc[g]
        if o is None or paths[g] is None:
            continue
        empty = np.flatnonzero(boards[g] == 2)
        if g % 5 == 0 and len(empty) >= 3:
            paths[g] = pick_cells(pair, rng, 3)[g]                                      # three plies
            kinds[g] = "three"
        elif g % 5 == 1:
            unvisited = [int(c) for c in empty if o.nodes[0].n[c] == 0]
            if unvisited:
                paths[g] = [unvisited[0]]
                kinds[g] = "unvisited"
    ply_paths(pair, paths)
    ex = raw.export()
    for g in range(G):
        if g % 5 == 2 and not ex["done"][g] and (boards[g] != 2).any():                 # a stone removed, same side to move
            b = sc.true_boards(ex)[g].reshape(-1).copy()
            b[np.flatnonzero(b != 2)[0]] = 2
            raw.import_boards(np.broadcast_to(b.reshape(N, N), (G, N, N)), np.full(G, ex["cur"][g], np.int8),
                              (np.arange(G) == g).astype(np.uint8))
            kinds[g] = "removed"
    amask = np.ones(G, np.uint8)
    amask[3] = 0
    pair.advance(8, root_mask=amask)
    for g, kind in kinds.items():
        o = pair.orc[g]
        if o is not None and g != 3:
            assert len(o.nodes) == 1 and o.s == 0 and o.nodes[0].flag == mcts.UNEXPANDED, (g, kind)
    assert pair.orc[3] is None
    # a move whose edge was visited while the pool was full: the child was never stored
    pair = Pair(raw_batch(4, 16, 6, 0, rng, fill=0.9), 6, 0, 3)
    pair.search(30)
    paths, hit = [], 0
    for o in pair.orc:
        full = [] if o is None else [int(c) for c in np.flatnonzero((o.nodes[0].n > 0) & (o.nodes[0].child < 0))] \
            if o.nodes[0].flag == mcts.EXPANDED else []
        paths.append(full[:1] or None)
        hit += bool(full)
    assert hit > 0
    ply_paths(pair, paths)
    pair.advance(1)
    for o, p in zip(pair.orc, paths):
        if p and o is not None:
            assert len(o.nodes) == 1 and o.s == 0


def test_a_pending_select_is_cleared():
    """advance clears a split-form leaf that select left pending: the next expand changes nothing."""
    N, G = 5, 9
    rng = np.random.default_rng(8)
    pair = Pair(raw_batch(N, G, 2, 1, rng), 2, 1, 60)
    pair.split(20, rng)
    pair.e.select()
    for o in pair.orc:
        if o is not None:
            o.select()
    ply_paths(pair, pick_cells(pair, rng, 1))
    pair.advance(3)
    root_bytes = int(pair.e.tree[40:48].view(np.int64)[0])
    for g in range(G):
        assert pair.e.tree[128 + g * root_bytes:].view(np.int32)[5] == 0                # meta[5]: pending
    snap = pair.e.tree.copy()
    pair.e.expand(np.ones((G, N * N), np.float32), np.zeros(G, np.float32))
    assert np.array_equal(snap, pair.e.tree)
    pair.split(10, rng)
    pair.check()


def test_used_is_the_reachable_count_and_the_pool_refills():
    N, G, M = 5, 10, 50
    rng = np.random.default_rng(9)
    pair = Pair(raw_batch(N, G, 1, 0, rng, fill=0.9), 1, 0, M)
    pair.search(80)
    old = copy.deepcopy(pair.orc)
    paths = pick_cells(pair, rng, 1, explore=0.0)
    ply_paths(pair, paths)
    pair.advance(2)
    roots = mc.parse_tree(pair.e.tree, N, G)
    kept = 0
    for g, (o, p) in enumerate(zip(old, paths)):
        if o is None or not p or pair.orc[g] is None or o.nodes[0].child[p[0]] < 0:
            continue
        assert roots[g]["used"] == len(ma.reachable(o, int(o.nodes[0].child[p[0]])))
        kept += roots[g]["used"] > 1
    assert kept > 0
    pair.search(80)
    pair.check()
    used = pair.e.root()[3]
    assert (used[[o is not None for o in pair.orc]] == M).any()


def test_sharding_does_not_change_the_advance():
    N, G, H = 5, 16, 7
    rng = np.random.default_rng(12)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.7, 2, boards).astype(np.int8)
    out = []
    for off, n in ((0, G), (0, H), (H, G - H)):
        raw = EmuBatch(0, N, n, seed=5, game_offset=off, raw=True)
        raw.import_boards(boards[off:off + n], to_move[off:off + n])
        t = mcts_advance_emu.EmuMCTS(raw, 40)
        t.reset()
        for m in range(3):
            t.search(30, 2)
            raw.ply(t.root()[0].argmax(1).astype(np.int32))
            t.advance(first_playout=10 * m)
        t.search(10, 2)
        out.append(mc.parse_tree(t.tree, N, n))
    whole, lo, hi = out
    mc.assert_trees_equal(lo + hi, [mc.as_oracle(r) for r in whole])


# ---------------------------------------------------------------------------------------------- the C ABI without a GPU
def test_abi_argument_checks_without_a_gpu():
    L = _native.lib()
    p = ctypes.c_void_p(4096)
    assert L.hexb_mcts_advance(None, None, 0, 0, None, None) == -1
    assert L.hexb_mcts_advance(None, p, 1 << 20, 0, None, None) == -1
    assert L.hexb_version() == (1 << 16) | 5


def test_emulated_advance_on_a_foreign_buffer_writes_nothing():
    rng = np.random.default_rng(1)
    raw = raw_batch(5, 6, 1, 1, rng)
    t = mcts_advance_emu.EmuMCTS(raw, 20)
    t.advance(first_playout=5)                                                        # never initialised
    assert not t.tree.any()
    other = raw_batch(5, 7, 1, 1, rng)
    u = mcts_advance_emu.EmuMCTS(other, 20)
    u.reset()
    u.search(10, 2)
    t.tree = u.tree.copy()                                                            # G differs
    t.advance(first_playout=5)
    assert np.array_equal(t.tree, u.tree)
