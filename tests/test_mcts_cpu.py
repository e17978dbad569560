"""CPU: the batched tree search (hexb_mcts_*) without a GPU - its device code (csrc/hexb_mcts.cuh) run by the host emulator against
the oracle (oracle/mcts.py) bit for bit over the whole tree, the oracle's own consistency, the consequences of the definition
(split calls, one simulation = playouts, sharding), the split form's leaf observations against copy_games + ply + encode, and the
argument checks of the C ABI."""
import ctypes

import numpy as np
import pytest

from emu.emu import EmuBatch, EmuMCTS, copy_games, playouts
from oracle import mcts, playout
from hex_gym_env_b200 import _native
import mcts_common as mc
import search_common as sc


def env_batch(N, G, seed, variant, agent_mode, opp_first, steps=None, auto_reset=True, reset_mask=None, game_offset=0):
    env = EmuBatch(variant, N, G, seed=seed, agent_mode=agent_mode, opponent_first=opp_first, auto_reset=auto_reset,
                   game_offset=game_offset)
    env.reset(reset_mask)
    for _ in range(sc.env_steps(N) if steps is None else steps):
        env.step()
    return env


def raw_batch(N, G, seed, variant, rng, game_offset=0):
    raw = EmuBatch(variant, N, G, seed=seed, game_offset=game_offset, raw=True)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.5, 2, boards).astype(np.int8)   # sparser: longer games
    raw.import_boards(boards, to_move)
    return raw


def fused(batch, seed, game_offset, variant, max_nodes, S, P, c_puct=1.5, fpu=0.25, first=3, root_mask=None, calls=(None,)):
    """The emulated tree after S simulations (in the given split of calls) and the oracle's trees after the same."""
    t = EmuMCTS(batch, max_nodes, c_puct, fpu)
    t.reset(root_mask, first)
    for k in (calls if calls != (None,) else (S,)):
        t.search(k, P)
    orc = mc.oracle_trees(batch.export(), seed, game_offset, variant, max_nodes, c_puct, fpu, first, root_mask)
    for o in orc:
        for _ in range(S if o is not None else 0):
            o.simulate(P)
    return t, orc


def split(batch, seed, variant, max_nodes, S, rng, c_puct=1.1, fpu=-0.2, root_mask=None, check_obs=None, live=None):
    """S select / expand rounds with seeded priors and values on the emulator and the oracle; leaf obs, masks and pending flags
    compared every round. live: the games ever reset (an export does not show it), None = all."""
    t = EmuMCTS(batch, max_nodes, c_puct, fpu)
    t.reset(root_mask)
    om = root_mask if live is None else (live if root_mask is None else root_mask & live)
    orc = mc.oracle_trees(batch.export(), seed, 0, variant, max_nodes, c_puct, fpu, 0, om)
    G, C = batch.G, batch.C
    for _ in range(S):
        obs, mask, pending = t.select()
        for g, o in enumerate(orc):
            want = o.select() if o is not None else None
            assert pending[g] == (want is not None), g
            if want is not None:
                assert np.array_equal(obs[g], want[0]) and np.array_equal(mask[g], want[1]), g
        if check_obs is not None:
            check_obs(orc, obs, mask, pending)
        priors = rng.dirichlet(np.ones(C), size=G).astype(np.float32)
        values = rng.uniform(-1, 1, size=G).astype(np.float32)
        t.expand(priors, values)
        for g, o in enumerate(orc):
            if o is not None and pending[g]:
                o.expand(priors[g], values[g])
    return t, orc


def check_tree(t, orc):
    mc.assert_trees_equal(mc.parse_tree(t.tree, t.batch.N, t.batch.G), orc)


# ---------------------------------------------------------------------------------------------- the oracle on its own
def walk(o):
    """(node, true board) for every node of an oracle tree."""
    out, stack = [], [(0, o.board.copy(), 0)]
    while stack:
        k, board, d = stack.pop()
        out.append((k, board, d))
        nd = o.nodes[k]
        if nd.flag == mcts.EXPANDED:
            for c in np.flatnonzero(nd.child >= 0):
                b = board.copy()
                b[c] = o.mover(d)
                stack.append((int(nd.child[c]), b, d + 1))
    return out


@pytest.mark.parametrize("N", (3, 4, 5))
def test_oracle_is_consistent(N):
    """Root visits sum to Nn(root) - 1; every node is reached once; terminal flags are exactly the nodes whose last move
    connected its player's edges; each node's Nn = 1 + the visits of its edges (a leaf's re-evaluations included)."""
    rng = np.random.default_rng(N)
    raw = raw_batch(N, 6, 9, 0, rng)
    _, orc = fused(raw, 9, 0, 0, 200, 60, 2)
    for o in orc:
        if o is None:
            continue
        assert int(o.nodes[0].n.sum()) == o.nodes[0].nn - 1
        seen = walk(o)
        assert sorted(k for k, _, _ in seen) == list(range(len(o.nodes)))
        for k, board, d in seen:
            nd = o.nodes[k]
            if k > 0:
                assert (nd.flag == mcts.TERMINAL) == playout.connects(board.reshape(N, N), o.mover(d - 1)), k
            if nd.flag == mcts.EXPANDED and (board == 2).any():
                assert nd.nn == 1 + int(nd.n.sum()), k


# ---------------------------------------------------------------------------------------------- emulator == oracle
@pytest.mark.parametrize("N", (3, 4, 5, 7, 9))
def test_fused_search_matches_the_oracle(N):
    """Env handles of every kind (WHITE agents stored transposed) and raw handles of both variants, ragged G, P = 3 playouts."""
    rng = np.random.default_rng(10 + N)
    S = 40 if N <= 5 else 24
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 50 * N + 10 * variant + agent_mode
        env = env_batch(N, 5, seed, variant, agent_mode, opp_first)
        check_tree(*fused(env, seed, 0, variant, 4 * S, S, 3))
    for variant in (0, 1):
        raw = raw_batch(N, 7, 77, variant, rng, game_offset=5)
        check_tree(*fused(raw, 77, 5, variant, 4 * S, S, 2, first=2 ** 32 - 20))   # playout indices wrap mod 2^32


def test_fused_search_13x13():
    env = env_batch(13, 3, 4, 1, 2, False, steps=20)
    check_tree(*fused(env, 4, 0, 1, 64, 12, 2))


def test_inactive_roots_and_a_full_pool():
    """Finished, never reset and masked-off roots stay untouched (nodes_used 0); max_nodes < S + 1 fills the pool."""
    N, G = 5, 37
    reset = np.ones(G, np.uint8)
    reset[::5] = 0
    env = env_batch(N, G, 8, 1, 2, False, steps=9, auto_reset=False, reset_mask=reset)
    ex = env.export()
    done = ex["done"].astype(bool)
    assert done.any() and not done.all()
    mask = reset.copy()
    mask[1::4] = 0
    t, orc = fused(env, 8, 0, 1, 9, 30, 2, root_mask=mask)
    check_tree(t, orc)
    visits, q, value, used = t.root()
    active = (mask == 1) & ~done
    assert ((used > 0) == active).all()
    assert (visits[~active] == 0).all() and (value[~active] == 0).all()
    assert (used[active] == 9).any()                                                  # the pool filled up
    for g in np.flatnonzero(active):
        v, qq, val = orc[g].root()
        assert np.array_equal(visits[g], v) and np.array_equal(q[g].view(np.uint32), qq.view(np.uint32))
        assert np.float32(value[g]).view(np.uint32) == np.float32(val).view(np.uint32)


@pytest.mark.parametrize("N", (3, 4, 5, 7, 9))
def test_split_search_matches_the_oracle(N):
    rng = np.random.default_rng(20 + N)
    S = 30 if N <= 5 else 20
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 60 * N + 10 * variant + agent_mode
        env = env_batch(N, 5, seed, variant, agent_mode, opp_first)
        check_tree(*split(env, seed, variant, 4 * S, S, rng))
    for variant in (0, 1):
        raw = raw_batch(N, 6, 7, variant, rng)
        check_tree(*split(raw, 7, variant, S // 2, S, rng))                           # the pool fills up


def test_split_search_13x13_and_inactive_roots():
    rng = np.random.default_rng(13)
    env = env_batch(13, 3, 5, 0, 0, True, steps=20)
    check_tree(*split(env, 5, 0, 32, 10, rng))
    N, G = 5, 19
    live = (np.arange(G) % 4 != 0).astype(np.uint8)
    env = env_batch(N, G, 6, 1, 2, False, steps=9, auto_reset=False, reset_mask=live)
    mask = (np.arange(G) % 3 != 0).astype(np.uint8)
    check_tree(*split(env, 6, 1, 12, 25, rng, root_mask=mask, live=live))


# ---------------------------------------------------------------------------------------------- consequences of the definition
def test_search_calls_add_up():
    """search(a); search(b) equals search(a + b): the same bytes for every root."""
    env = env_batch(6, 9, 2, 1, 2, False)
    a = EmuMCTS(env, 80, 1.3, 0.0)
    b = EmuMCTS(env, 80, 1.3, 0.0)
    a.reset(first_playout=11)
    b.reset(first_playout=11)
    a.search(17, 4)
    a.search(29, 4)
    b.search(46, 4)
    assert np.array_equal(a.tree, b.tree)


def test_one_simulation_is_the_playout_value():
    """After search(1) value = (2 * playouts(P, first) - P) / P and every root visit count is 0."""
    P, first = 37, 9
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        env = env_batch(7, 20, 3 + variant, variant, agent_mode, opp_first)
        t = EmuMCTS(env, 10)
        t.reset(first_playout=first)
        t.search(1, P)
        visits, q, value, used = t.root()
        wins = playouts(env, P, first)
        ok = wins >= 0
        assert ((used > 0) == ok).all()
        want = (np.float32(2) * wins.astype(np.float32) - np.float32(P)) / np.float32(P)
        assert np.array_equal(value[ok], want[ok].astype(np.float32)) and (visits == 0).all()


def test_results_do_not_depend_on_sharding():
    """Two shards (game_offset) search what one batch searches: the streams key on the global game index."""
    N, G, H = 5, 24, 10
    rng = np.random.default_rng(3)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.6, 2, boards).astype(np.int8)
    trees = []
    for off, n in ((0, G), (0, H), (H, G - H)):
        raw = EmuBatch(1, N, n, seed=21, game_offset=off, raw=True)
        raw.import_boards(boards[off:off + n], to_move[off:off + n])
        t = EmuMCTS(raw, 40)
        t.reset()
        t.search(30, 3)
        trees.append(mc.parse_tree(t.tree, N, n))
    whole, lo, hi = trees
    mc.assert_trees_equal(lo + hi, [mc.as_oracle(r) for r in whole])


def test_split_leaf_obs_is_copy_ply_encode():
    """Each pending leaf's obs and mask equal encode(view 1) of a raw copy of the root with the path's moves played by ply."""
    rng = np.random.default_rng(5)
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        N, G = 6, 8
        env = env_batch(N, G, 30 + variant, variant, agent_mode, opp_first)

        def check(orc, obs, mask, pending):
            raw = EmuBatch(variant, N, G, raw=True)
            copy_games(raw, env)
            paths = [o.leaf["cells"][1:] if o is not None and o.leaf is not None else [] for o in orc]
            for d in range(max(len(p) for p in paths)):
                acts = np.full(G, -1, np.int32)
                for g, p in enumerate(paths):
                    if d < len(p):
                        acts[g] = mcts.action(variant, orc[g].mover(d), N, p[d])
                raw.ply(acts)
            o1, m1 = raw.encode(1)
            rows = pending == 1
            assert np.array_equal(obs[rows], o1[rows]) and np.array_equal(mask[rows], m1[rows])

        split(env, 30 + variant, variant, 60, 25, rng, check_obs=check)


# ---------------------------------------------------------------------------------------------- the C ABI without a GPU
def test_abi_argument_checks_without_a_gpu():
    L = _native.lib()
    p, n = ctypes.c_void_p(4096), ctypes.c_size_t(0)
    assert L.hexb_mcts_tree_bytes(None, 10, ctypes.byref(n)) == -1
    assert L.hexb_mcts_init(None, p, 1 << 20, 10, 1.0, 0.0, 0, None, None) == -1
    assert L.hexb_mcts_search(None, p, 1 << 20, 1, 1, None) == -1
    assert L.hexb_mcts_select(None, p, 1 << 20, p, p, p, None) == -1
    assert L.hexb_mcts_expand(None, p, 1 << 20, p, p, None) == -1
    assert L.hexb_mcts_root(None, p, 1 << 20, p, p, p, p, None) == -1
    assert L.hexb_version() == (1 << 16) | 5                                           # additive: the version stays 1.5


def test_emulated_calls_on_a_foreign_buffer_write_nothing():
    """A buffer that holds no tree of this batch (never initialised, or another batch's) is left alone."""
    env = env_batch(5, 6, 1, 1, 2, False)
    t = EmuMCTS(env, 20)
    t.search(5, 2)                                                                    # before any reset
    t.select()
    t.expand(np.ones((6, 25), np.float32), np.zeros(6, np.float32))
    assert not t.tree.any()
    other = env_batch(5, 7, 1, 1, 2, False)
    u = EmuMCTS(other, 20)
    u.reset()
    t.tree = u.tree.copy()                                                            # G differs
    t.search(5, 2)
    assert np.array_equal(t.tree, u.tree)
