"""CPU: the tree search's float edges and its playout key at the top of their ranges, run by the host emulator (the device code of
csrc/hexb_mcts.cuh) against the oracle (oracle/mcts.py) - the ranking of NaN and signed-zero scores (include/hexb.h), priors and
values at the float32 limits, c_puct / fpu of 0, tiny, huge and infinite size, and a game offset past 2^32 with playout indices
that wrap mod 2^32 part-way through a simulation's playouts."""
import numpy as np
import pytest

from emu.emu import EmuBatch, EmuMCTS
from oracle import mcts
import mcts_common as mc
import search_common as sc

F = np.float32
pytestmark = pytest.mark.filterwarnings("ignore::RuntimeWarning")   # the oracle's float32 overflows and NaNs are the point here


def raw_pair(N, G, seed, variant, rng, game_offset=0, fill=0.5):
    raw = EmuBatch(variant, N, G, seed=seed, game_offset=game_offset, raw=True)
    boards, to_move = sc.random_boards(rng, G, N)
    boards = np.where(rng.uniform(size=boards.shape) < fill, 2, boards).astype(np.int8)
    raw.import_boards(boards, to_move)
    return raw


def split_rounds(t, orc, S, inputs):
    """S select / expand rounds on the emulator and the oracle; leaf rows and pending flags compared every round."""
    G = t.batch.G
    for _ in range(S):
        obs, mask, pending = t.select()
        for g, o in enumerate(orc):
            want = o.select() if o is not None else None
            assert pending[g] == (want is not None), g
            if want is not None:
                assert np.array_equal(obs[g], want[0]) and np.array_equal(mask[g], want[1]), g
        priors, values = inputs(mask)
        t.expand(priors, values)
        for g, o in enumerate(orc):
            if o is not None and pending[g]:
                o.expand(priors[g], values[g])
    assert len(orc) == G


def check(t, orc):
    mc.assert_trees_equal(mc.parse_tree(t.tree, t.batch.N, t.batch.G), orc)
    got = t.root()
    for g, o in enumerate(orc):
        if o is not None:
            v, q, val = o.root()
            mc.assert_root_outputs_equal([x[g] for x in got], (v, q, val, len(o.nodes)))


# ---------------------------------------------------------------------------------------------- the ranking rule
def test_key_ranks_nan_below_every_number_and_ties_signed_zeros():
    nans = [np.array([b], np.uint32).view(np.float32)[0] for b in (0x7fffffff, 0xffc00000, 0x7fc00000, 0xff800001)]
    lowest = mcts.key(F(-np.inf), 100)
    for x in nans:
        assert np.isnan(x)
        assert 0 < mcts.key(x, 0) < lowest                          # below -inf, still a key (0 = no empty cell)
        assert mcts.key(x, 3) > mcts.key(nans[0], 4)                # NaN against NaN: the lower cell wins
    assert mcts.key(F(-0.0), 3) > mcts.key(F(0.0), 4) > mcts.key(F(-1e-45), 0)
    assert mcts.key(F(0.0), 3) > mcts.key(F(-0.0), 4)
    assert mcts.key(F(np.inf), 9) > mcts.key(F(3e38), 0) > mcts.key(F(-3e38), 0) > lowest


def one_root(N, board, to_move, c_puct, fpu):
    """A raw one-game batch holding `board`, and the emulator's and the oracle's trees on it."""
    raw = EmuBatch(1, N, 1, seed=3, raw=True)
    raw.import_boards(board[None], np.array([to_move], np.int8))
    t = EmuMCTS(raw, 64, c_puct, fpu)
    t.reset()
    o = mc.oracle_trees(raw.export(), 3, 0, 1, 64, c_puct, fpu, 0)
    return t, o


@pytest.mark.parametrize("nan", (0x7fc00000, 0xffc00000))
def test_a_nan_child_gets_no_more_visits(nan):
    """After a NaN value is backed up through one root edge, that edge is never selected again while another empty cell has a
    number for Q + U. Both NaN signs: the host keeps the sign the backup gives the NaN, and the bits must not rank it."""
    N = 4
    board = np.full((N, N), 2, np.int8)
    t, orc = one_root(N, board, 0, 1.0, 0.0)
    first = [True]

    def inputs(mask):
        priors = np.full((1, N * N), 1.0 / (N * N), np.float32)
        value = np.array([0.5], np.float32)
        if first[0]:
            first[0] = False
        elif t.root()[0][0].sum() == 0:                             # the first child leaf: its value is NaN
            value = np.array([nan], np.uint32).view(np.float32)
        return priors, value

    split_rounds(t, orc, 40, inputs)
    check(t, orc)
    visits, q = t.root()[0][0], t.root()[1][0]
    assert np.isnan(q[0]) and visits[0] == 1                        # cell 0 (the lowest) was taken first, then never again
    assert (visits[1:] > 0).sum() >= 10


def test_all_nan_scores_take_the_lowest_empty_cell():
    """c_puct = inf and zero priors: every U is inf * 0 = NaN, so every cell ranks the same and the lowest empty cell wins."""
    N = 5
    rng = np.random.default_rng(1)
    board = np.where(rng.uniform(size=(N, N)) < 0.3, 1, 2).astype(np.int8)
    board[0, 0] = 1
    t, orc = one_root(N, board, 0, np.inf, 0.0)
    split_rounds(t, orc, 12, lambda mask: (np.zeros((1, N * N), np.float32), rng.uniform(-1, 1, 1).astype(np.float32)))
    check(t, orc)
    visits = t.root()[0][0]
    lowest = int(np.flatnonzero(board.reshape(-1) == 2)[0])
    assert visits[lowest] == visits.sum() == 11


def test_signed_zero_scores_tie_to_the_lowest_cell():
    """fpu = -0 and a prior of -0 give a Q + U of -0, a prior of +0 one of +0: a tie, so the lowest empty cell wins."""
    N = 4
    board = np.full((N, N), 2, np.int8)
    t, orc = one_root(N, board, 0, 1.0, -0.0)
    pri = np.zeros((1, N * N), np.float32)
    pri[0, 0] = -0.0
    split_rounds(t, orc, 2, lambda mask: (pri, np.zeros(1, np.float32)))
    check(t, orc)
    assert t.root()[0][0][0] == 1 and t.root()[0][0].sum() == 1


# ---------------------------------------------------------------------------------------------- float edges
@pytest.mark.parametrize("c_puct, fpu", mc.EDGE_SETTINGS)
def test_float_edges_match_the_oracle(c_puct, fpu):
    """Split form with priors and values from mcts_common.EDGE_PRIORS / EDGE_VALUES, both variants, a pool that fills."""
    rng = np.random.default_rng(mc.EDGE_SETTINGS.index((c_puct, fpu)))
    for variant, N in ((0, 4), (1, 5)):
        raw = raw_pair(N, 6, 11, variant, rng)
        t = EmuMCTS(raw, 20, c_puct, fpu)
        t.reset()
        orc = mc.oracle_trees(raw.export(), 11, 0, variant, 20, c_puct, fpu, 0)
        split_rounds(t, orc, 30, lambda mask: mc.edge_inputs(rng, raw.G, raw.C))
        check(t, orc)


# ---------------------------------------------------------------------------------------------- the playout key
@pytest.mark.parametrize("N", (3, 5, 7))
def test_playout_key_past_2_to_the_32(N):
    """game_offset = 12345678901 (the key's high word is not 0) and first_playout = 2^32 - 40 with P = 33: the playout index wraps
    mod 2^32 inside the second simulation's playouts. Env handles and raw handles of both variants."""
    off, first, P, S = 12345678901, 2 ** 32 - 40, 33, 8
    rng = np.random.default_rng(N)
    batches = [(raw_pair(N, 4, 5, v, rng, game_offset=off), v) for v in (0, 1)]
    env = EmuBatch(1, N, 3, seed=5, game_offset=off, agent_mode=2)
    env.reset()
    for _ in range(sc.env_steps(N) // 2):
        env.step()
    batches.append((env, 1))
    for b, variant in batches:
        t = EmuMCTS(b, S + 1, 1.25, 0.0)
        t.reset(first_playout=first)
        t.search(S, P)
        orc = mc.oracle_trees(b.export(), 5, off, variant, S + 1, 1.25, 0.0, first)
        for o in orc:
            for _ in range(S if o is not None else 0):
                o.simulate(P)
        check(t, orc)
