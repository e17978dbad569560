"""CPU: bridge-reply playouts (include/hexb.h, HEXB_PLAYOUT_BRIDGE) without a GPU - the restated rule (bridge_oracle.py) on
hand-built positions and over seeded playouts, the device code (csrc/hexb_search.cuh, csrc/hexb_mcts.cuh) run by the host emulator
against it bit for bit (playouts_policy wins and whole search_policy trees), and the argument checks of the new C ABI entries."""
import ctypes

import numpy as np
import pytest

import bridge_oracle as bo
import mcts_common as mc
import search_common as sc
from emu import bridge_emu, mcts_emu, search_emu
from emu.emu import EmuBatch
from oracle import playout
from hex_gym_env_b200 import PLAYOUT_BRIDGE, PLAYOUT_RANDOM, _native

B, W, E = bo.BLACK, bo.WHITE, bo.EMPTY


def board_with(N, stones):
    """A true N x N board (0 BLACK, 1 WHITE, 2 EMPTY) with stones {(y, x): colour}."""
    b = np.full((N, N), E, np.int8)
    for (y, x), c in stones.items():
        b[y, x] = c
    return b


def cell(N, y, x):
    return y * N + x


# ---------------------------------------------------------------------------------------------- the rule on its own
def test_policy_codes_are_the_header_s():
    assert (PLAYOUT_RANDOM, PLAYOUT_BRIDGE) == (bo.PLAYOUT_RANDOM, bo.PLAYOUT_BRIDGE) == (0, 1)
    with open(_native.HEADER) as f:
        text = f.read()
    assert "#define HEXB_PLAYOUT_RANDOM 0" in text and "#define HEXB_PLAYOUT_BRIDGE 1" in text


def test_d_is_the_reference_neighbourhood_in_cyclic_order():
    """D holds the six neighbours of the reference (3x3 window minus (-1,-1) and (+1,+1)), and the common neighbours of c and
    c + D[i] are exactly c + D[i-1] and c + D[i+1]."""
    assert sorted(bo.D) == sorted(playout.NEIGHBOURS)
    nb = set(playout.NEIGHBOURS)
    for i, (dy, dx) in enumerate(bo.D):
        common = {(ay, ax) for ay, ax in nb if (ay - dy, ax - dx) in nb}
        assert common == {bo.D[i - 1], bo.D[(i + 1) % 6]}, i


@pytest.mark.parametrize("mover", (B, W))
@pytest.mark.parametrize("i", range(6))
def test_interior_bridge_in_each_direction(i, mover):
    """The opponent intrudes at prev into the bridge of the mover's stones prev + D[i-1], prev + D[i+1]: the reply is prev + D[i].
    The same stones of the other colour give nothing."""
    N, py, px = 7, 3, 3
    (ay, ax), (by, bx), (ey, ex) = bo.D[i - 1], bo.D[(i + 1) % 6], bo.D[i]
    for owner in (mover, 1 - mover):
        b = board_with(N, {(py, px): 1 - mover, (py + ay, px + ax): owner, (py + by, px + bx): owner})
        want = [cell(N, py + ey, px + ex)] if owner == mover else []
        assert bo.bridge_replies(b, mover, cell(N, py, px)) == want, (i, owner)


def edge_cases(N):
    """(owner, stone, carrier a, carrier b) for edge bridges on all four edges: the stone's two neighbours on the owner's edge."""
    out = []
    for x in (0, 1, 2, N - 2):
        out.append((B, (1, x), (0, x), (0, x + 1)))                 # top: (1, x) touches (0, x), (0, x + 1)
    for x in (1, 2, 3, N - 2, N - 1):
        out.append((B, (N - 2, x), (N - 1, x - 1), (N - 1, x)))     # bottom
    for y in (0, 1, 2, N - 2):
        out.append((W, (y, 1), (y, 0), (y + 1, 0)))                 # left
    for y in (1, 2, 3, N - 2, N - 1):
        out.append((W, (y, N - 2), (y - 1, N - 1), (y, N - 1)))     # right
    return out


@pytest.mark.parametrize("N", (5, 7, 11))
def test_edge_bridges_on_all_four_edges(N):
    """A stone on the second row (column) with its two edge cells empty is bridged to its owner's edge: an intrusion in either
    carrier cell is answered in the other. The same stone of the colour that does not own that edge gets no reply (unless it
    is also on the second line of that colour's own edge, next to a corner)."""
    nb = set(playout.NEIGHBOURS)
    for owner, s, a, b in edge_cases(N):
        assert (a[0] - s[0], a[1] - s[1]) in nb and (b[0] - s[0], b[1] - s[1]) in nb
        along = s[1] if owner == B else s[0]
        for prev, other in ((a, b), (b, a)):
            for mover in (B, W):
                if mover != owner and along in (1, N - 2):
                    continue
                bd = board_with(N, {s: mover, prev: 1 - mover})
                want = [cell(N, *other)] if mover == owner else []
                assert bo.bridge_replies(bd, mover, cell(N, *prev)) == want, (owner, s, prev, mover)


def test_corner_points_belong_to_no_one():
    """A stone at (1, N-1) touches (0, N-1) and the corner point (-1, N); an intrusion at (0, N-1) gets no edge reply."""
    N = 7
    for mover in (B, W):
        bd = board_with(N, {(1, N - 1): mover, (0, N - 1): 1 - mover})
        assert bo.bridge_replies(bd, mover, cell(N, 0, N - 1)) == []


def test_two_and_three_candidates_choose_in_row_major_order():
    """The mover's stones at D[1], D[3], D[5] around the intrusion prev make three bridges through it (replies D[0], D[2], D[4]);
    with D[4] taken by the opponent two remain. Ply 0 plays R[int(u * |R|)] in row-major order, and every candidate is taken by
    some playout."""
    N, py, px = 7, 3, 3
    pc = cell(N, py, px)
    at = lambda d: (py + bo.D[d][0], px + bo.D[d][1])
    for mover in (B, W):
        for taken, reply_dirs in ((None, (0, 2, 4)), (4, (0, 2))):
            stones = {at(d): mover for d in (1, 3, 5)}
            stones[(py, px)] = 1 - mover
            if taken is not None:
                stones[at(taken)] = 1 - mover
            bd = board_with(N, stones)
            R = bo.bridge_replies(bd, mover, pc)
            assert R == sorted(cell(N, *at(d)) for d in reply_dirs) and len(R) == len(reply_dirs)
            hit = set()
            for p in range(64):
                c, u, rr, _ = bo.playout_plies(bd, mover, 9, 4, p, bo.PLAYOUT_BRIDGE, pc)[0]
                assert rr == R and c == R[bo.choice(u, len(R))]
                hit.add(c)
            assert hit == set(R)


def test_occupied_carrier_gives_no_reply():
    """The other carrier cell already holds a stone (either colour): no reply."""
    N, py, px = 7, 3, 3
    for mover in (B, W):
        for i in range(6):
            (ay, ax), (by, bx), (ey, ex) = bo.D[i - 1], bo.D[(i + 1) % 6], bo.D[i]
            for filler in (B, W):
                bd = board_with(N, {(py, px): 1 - mover, (py + ay, px + ax): mover, (py + by, px + bx): mover,
                                    (py + ey, px + ex): filler})
                assert bo.bridge_replies(bd, mover, cell(N, py, px)) == []


@pytest.mark.parametrize("N", (3, 5, 7, 11))
def test_seeded_playouts_follow_the_rule(N):
    """Over seeded playouts from random positions: a ply with an empty reply set plays the cell the random policy would play on
    that board with that u; every other ply plays R[int(u * |R|)]. Replies do happen. The random policy's plies equal
    oracle/playout.py's, and a playout without any reply is the random playout."""
    rng = np.random.default_rng(40 + N)
    boards, to_move = sc.random_boards(rng, 8, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.5, E, boards).astype(np.int8)
    replied = 0
    for g in range(8):
        b0, t = boards[g], int(to_move[g])
        for p in range(6):
            prev = None if p % 2 == 0 else int(rng.integers(0, N * N))
            plies = bo.playout_plies(b0, t, 17, g, p, bo.PLAYOUT_BRIDGE, prev)
            for c, u, R, rnd in plies:
                if R:
                    replied += 1
                    assert c == R[bo.choice(u, len(R))]
                else:
                    assert c == rnd
            assert sorted(c for c, _, _, _ in plies) == sorted(np.flatnonzero(b0.reshape(-1) == E).tolist())
            rand = [c for c, _, _, _ in bo.playout_plies(b0, t, 17, g, p)]
            assert rand == playout.playout_cells(b0, t, 17, g, p)
            if not any(R for _, _, R, _ in plies):
                assert [c for c, _, _, _ in plies] == rand
    assert replied > 0


# ---------------------------------------------------------------------------------------------- emulator == restated rule
def env_batch(N, G, seed, variant, agent_mode, opp_first, steps=None, auto_reset=True, game_offset=0):
    env = EmuBatch(variant, N, G, seed=seed, agent_mode=agent_mode, opponent_first=opp_first, auto_reset=auto_reset,
                   game_offset=game_offset)
    env.reset()
    for _ in range(sc.env_steps(N) if steps is None else steps):
        env.step()
    return env


def raw_batch(N, G, seed, variant, rng, game_offset=0):
    raw = EmuBatch(variant, N, G, seed=seed, game_offset=game_offset, raw=True)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < 0.5, E, boards).astype(np.int8)
    raw.import_boards(boards, to_move)
    return raw


def oracle_wins(batch, seed, game_offset, first, P, policy, mask=None):
    ex = batch.export()
    boards = sc.true_boards(ex)
    out = np.full(batch.G, -1, np.int32)
    for g in range(batch.G):
        if ex["done"][g] or (mask is not None and not mask[g]):
            continue
        out[g] = bo.wins(boards[g], int(ex["cur"][g]), seed, game_offset + g, first, P, policy)
    return out


@pytest.mark.parametrize("N", (3, 4, 5, 7, 9, 13))
def test_emulated_bridge_playouts_match_the_rule(N):
    """Env games of both variants (WHITE agents stored transposed) and raw games of both variants, P = 37, first_playout > 0:
    wins of playouts_policy(bridge) equal the restated rule bit for bit."""
    rng = np.random.default_rng(N)
    G, P, first = 3, 37, 5
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 1000 * N + 10 * variant + agent_mode
        env = env_batch(N, G, seed, variant, agent_mode, opp_first)
        got = bridge_emu.playouts(env, P, first, policy=PLAYOUT_BRIDGE)
        assert np.array_equal(got, oracle_wins(env, seed, 0, first, P, bo.PLAYOUT_BRIDGE)), (variant, agent_mode)
    for variant in (0, 1):
        raw = raw_batch(N, G, 77, variant, rng, game_offset=5)
        got = bridge_emu.playouts(raw, P, first, policy=PLAYOUT_BRIDGE)
        assert np.array_equal(got, oracle_wins(raw, 77, 5, first, P, bo.PLAYOUT_BRIDGE)), variant


def test_emulated_bridge_playouts_skip_finished_masked_and_unreset_games():
    N, G = 5, 64
    fresh = EmuBatch(1, N, G, seed=3, agent_mode=2)
    assert (bridge_emu.playouts(fresh, 8, policy=PLAYOUT_BRIDGE) == -1).all()
    env = env_batch(N, G, 3, 1, 2, False, steps=7, auto_reset=False)
    done = env.export()["done"].astype(bool)
    assert done.any() and not done.all()
    mask = np.ones(G, np.uint8)
    mask[::3] = 0
    w = bridge_emu.playouts(env, 8, 0, mask, policy=PLAYOUT_BRIDGE)
    assert ((w == -1) == (done | (mask == 0))).all()
    assert np.array_equal(w, oracle_wins(env, 3, 0, 0, 8, bo.PLAYOUT_BRIDGE, mask))


def test_bridge_policy_changes_some_results_and_random_is_unchanged():
    """The two policies differ somewhere on a mid-game batch, and policy 0 is hexb_playouts (the oracle's random playouts, and
    the emulated hexb_playouts / hexb_mcts_search of search_emu and mcts_emu byte for byte)."""
    env = env_batch(9, 16, 12, 1, 2, False)
    r = bridge_emu.playouts(env, 64, 3)
    assert np.array_equal(bridge_emu.playouts(env, 64, 3, policy=PLAYOUT_RANDOM), r)
    assert np.array_equal(r, search_emu.playouts(env, 64, 3))
    assert np.array_equal(r, oracle_wins(env, 12, 0, 3, 64, bo.PLAYOUT_RANDOM))
    assert not np.array_equal(bridge_emu.playouts(env, 64, 3, policy=PLAYOUT_BRIDGE), r)
    old, new = mcts_emu.EmuMCTS(env, 60, 1.3, 0.0), bridge_emu.EmuMCTS(env, 60, 1.3, 0.0)
    for t in (old, new):
        t.reset(first_playout=5)
    old.search(40, 3)
    new.search(40, 3, PLAYOUT_RANDOM)
    assert np.array_equal(old.tree, new.tree)


def fused(batch, seed, game_offset, variant, max_nodes, S, P, policy, c_puct=1.5, fpu=0.25, first=3, root_mask=None, calls=None):
    """The emulated tree after S simulations of search_policy (in the given split of calls) and the restated trees."""
    t = bridge_emu.EmuMCTS(batch, max_nodes, c_puct, fpu)
    t.reset(root_mask, first)
    for k in (calls or (S,)):
        t.search(k, P, policy)
    boards, ex = sc.true_boards(batch.export()), batch.export()
    orc = []
    for g in range(batch.G):
        ok = not ex["done"][g] and (root_mask is None or root_mask[g])
        orc.append(bo.RootTree(boards[g], int(ex["cur"][g]), max_nodes, c_puct, fpu, first, variant, seed, game_offset + g)
                   if ok else None)
    for o in orc:
        for _ in range(S if o is not None else 0):
            o.simulate(P, policy)
    return t, orc


def check_tree(t, orc):
    mc.assert_trees_equal(mc.parse_tree(t.tree, t.batch.N, t.batch.G), orc)


@pytest.mark.parametrize("N", (3, 4, 5, 7, 9, 13))
def test_emulated_bridge_search_matches_the_rule(N):
    """Whole trees of search_policy(bridge): env handles of every kind, raw handles of both variants (playout indices wrapping
    mod 2^32), ragged G, P = 3 and 2."""
    rng = np.random.default_rng(10 + N)
    S = 40 if N <= 5 else (24 if N <= 9 else 10)
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 50 * N + 10 * variant + agent_mode
        env = env_batch(N, 5 if N < 13 else 2, seed, variant, agent_mode, opp_first, steps=None if N < 13 else 20)
        check_tree(*fused(env, seed, 0, variant, 4 * S, S, 3, bo.PLAYOUT_BRIDGE))
    for variant in (0, 1):
        raw = raw_batch(N, 7 if N < 13 else 3, 77, variant, rng, game_offset=5)
        check_tree(*fused(raw, 77, 5, variant, 4 * S, S, 2, bo.PLAYOUT_BRIDGE, first=2 ** 32 - 20))


def test_emulated_bridge_search_masked_finished_unreset_and_full_pool():
    N, G = 5, 24
    env = EmuBatch(1, N, G, seed=6, agent_mode=2, auto_reset=False)
    reset_mask = np.ones(G, np.uint8)
    reset_mask[[1, 7]] = 0                                              # never reset: inactive
    env.reset(reset_mask)
    for _ in range(9):
        env.step()
    root_mask = np.ones(G, np.uint8)
    root_mask[::4] = 0
    ex = env.export()
    assert ex["done"].any()
    t, orc = fused(env, 6, 0, 1, 9, 30, 2, bo.PLAYOUT_BRIDGE, root_mask=root_mask & reset_mask)
    t2 = bridge_emu.EmuMCTS(env, 9, 1.5, 0.25)
    t2.reset(root_mask, 3)
    t2.search(30, 2, PLAYOUT_BRIDGE)
    assert np.array_equal(t.tree, t2.tree)                              # never-reset games are inactive without a mask
    check_tree(t, orc)
    assert any(o is not None and len(o.nodes) == 9 for o in orc)                  # a pool that filled up


def test_emulated_bridge_search_calls_add_up():
    """search(a); search(b) equals search(a + b) under the bridge policy: the same bytes for every root."""
    env = env_batch(6, 9, 2, 1, 2, False)
    a = bridge_emu.EmuMCTS(env, 80, 1.3, 0.0)
    b = bridge_emu.EmuMCTS(env, 80, 1.3, 0.0)
    a.reset(first_playout=11)
    b.reset(first_playout=11)
    a.search(17, 4, PLAYOUT_BRIDGE)
    a.search(29, 4, PLAYOUT_BRIDGE)
    b.search(46, 4, PLAYOUT_BRIDGE)
    assert np.array_equal(a.tree, b.tree)
    c = bridge_emu.EmuMCTS(env, 80, 1.3, 0.0)
    c.reset(first_playout=11)
    c.search(46, 4, PLAYOUT_RANDOM)
    assert not np.array_equal(c.tree, b.tree)


def test_emulated_bridge_search_first_simulation_is_the_playout_value():
    """Node 0's leaf has no previous move: after search(1) the root value is playouts_policy(bridge)'s."""
    P, first = 37, 9
    env = env_batch(7, 20, 3, 1, 2, False)
    t = bridge_emu.EmuMCTS(env, 10)
    t.reset(first_playout=first)
    t.search(1, P, PLAYOUT_BRIDGE)
    _, _, value, used = t.root()
    wins = bridge_emu.playouts(env, P, first, policy=PLAYOUT_BRIDGE)
    ok = wins >= 0
    want = (np.float32(2) * wins.astype(np.float32) - np.float32(P)) / np.float32(P)
    assert ((used > 0) == ok).all() and np.array_equal(value[ok], want[ok].astype(np.float32))


# ---------------------------------------------------------------------------------------------- the C ABI without a GPU
def test_abi_argument_checks_without_a_gpu():
    """Null handles and bad policy values are refused before any device work (the handle is never read for a bad policy)."""
    L = _native.lib()
    p = ctypes.c_void_p(4096)
    fake = ctypes.create_string_buffer(4096)
    h = ctypes.cast(fake, ctypes.c_void_p)
    assert L.hexb_playouts_policy(None, 8, 0, 0, None, p, None) == -1
    assert L.hexb_playouts_policy(None, 8, 0, 1, None, p, None) == -1
    assert L.hexb_mcts_search_policy(None, p, 1 << 20, 1, 1, 0, None) == -1
    assert L.hexb_mcts_search_policy(None, p, 1 << 20, 1, 1, 1, None) == -1
    for bad in (-1, 2, 3, 1 << 30):
        assert L.hexb_playouts_policy(h, 8, 0, bad, None, p, None) == -1, bad
        assert L.hexb_mcts_search_policy(h, p, 1 << 20, 1, 1, bad, None) == -1, bad
    assert L.hexb_version() == (1 << 16) | 5                            # additive: the version stays 1.5


def test_python_policy_checks_without_a_gpu():
    from hex_gym_env_b200.batch import _playout_policy
    assert _playout_policy(PLAYOUT_RANDOM) == 0 and _playout_policy(PLAYOUT_BRIDGE) == 1 and _playout_policy(np.int64(1)) == 1
    for bad in (-1, 2, "1", None, True, 0.5):
        with pytest.raises(ValueError):
            _playout_policy(bad)
    env = EmuBatch(1, 5, 2, raw=True)
    for bad in (-1, 2):
        with pytest.raises(ValueError):
            bridge_emu.playouts(env, 4, policy=bad)
        with pytest.raises(ValueError):
            bridge_emu.EmuMCTS(env, 4).search(1, 1, bad)
