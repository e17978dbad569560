"""CPU: the tree-search primitives (hexb_copy_games, hexb_playouts) without a GPU - their device code (csrc/hexb_search.cuh) run by
the host emulator against the playout oracle (oracle/playout.py), the oracle's full-board shortcut against the C oracle's own
win check, the env -> raw conversion against the source game's export, and the argument checks of the C ABI."""
import ctypes

import numpy as np
import pytest

from emu.emu import EmuBatch, copy_games, playouts
from oracle import hexref, playout
from hex_gym_env_b200 import _native
import search_common as sc

STATE_KEYS = ("regions", "region_counter", "cur", "done", "winner")


def env_batch(N, G, seed, variant, agent_mode, opponent_first, steps=None, auto_reset=True):
    env = EmuBatch(variant, N, G, seed=seed, agent_mode=agent_mode, opponent_first=opponent_first, auto_reset=auto_reset)
    env.reset()
    for _ in range(sc.env_steps(N) if steps is None else steps):
        env.step()
    return env


def oracle_wins(batch, seed, game_offset, first, P):
    ex = batch.export()
    boards = sc.true_boards(ex)
    out = np.full(batch.G, -1, np.int32)
    for g in range(batch.G):
        if ex["done"][g]:
            continue
        out[g] = playout.wins(boards[g], int(ex["cur"][g]), seed, game_offset + g, first, P)
    return out


@pytest.mark.parametrize("N", range(3, 20))
def test_emulated_playouts_match_the_oracle(N):
    """Env games of both variants (WHITE agents are stored transposed) and preset raw boards, either side to move, P = 37
    (not a multiple of 32), first_playout > 0: the kernel's per-game code equals the oracle bit for bit."""
    rng = np.random.default_rng(N)
    G, P, first = 3, 37, 5
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 1000 * N + 10 * variant + agent_mode
        env = env_batch(N, G, seed, variant, agent_mode, opp_first)
        assert np.array_equal(playouts(env, P, first), oracle_wins(env, seed, 0, first, P)), (variant, agent_mode)
    for variant in (0, 1):
        raw = EmuBatch(variant, N, G, seed=77, game_offset=5, raw=True)
        boards, to_move = sc.random_boards(rng, G, N)
        raw.import_boards(boards, to_move)
        assert np.array_equal(playouts(raw, P, first), oracle_wins(raw, 77, 5, first, P)), variant


def test_emulated_playouts_skip_finished_masked_and_unreset_games():
    N, G = 5, 64
    fresh = EmuBatch(1, N, G, seed=3, agent_mode=2)
    assert (playouts(fresh, 8) == -1).all()                       # never reset
    env = env_batch(N, G, 3, 1, 2, False, steps=7, auto_reset=False)
    done = env.export()["done"].astype(bool)
    assert done.any() and not done.all()
    mask = np.ones(G, np.uint8)
    mask[::3] = 0
    w = playouts(env, 8, 0, mask)
    assert ((w == -1) == (done | (mask == 0))).all()
    assert ((w >= 0) & (w <= 8))[~done & (mask == 1)].all()


def test_emulated_playouts_first_playout_offsets_the_streams():
    """Playouts [0, 40) in one call are the sum of [0, 17) and [17, 40)."""
    env = env_batch(7, 8, 11, 1, 2, False)
    assert np.array_equal(playouts(env, 40, 0), playouts(env, 17, 0) + playouts(env, 23, 17))


@pytest.mark.parametrize("N", (3, 4, 5, 8, 11))
def test_full_board_winner_is_the_reference_winner(N):
    """Each oracle playout's cell sequence replayed through the C oracle's raw HexGame plies until make_move reports a winner gives
    the same winner as the filled board's connectivity test."""
    rng = np.random.default_rng(100 + N)
    G = 12
    ref = hexref.RefBatch(hexref.KIND_GAME_A, N, G)
    ref.set_board(np.full((G, N, N), 2, np.int8), 0)
    for _ in range(int(rng.integers(0, N * N // 2))):   # random plies from the empty board: positions nobody has won yet
        ex = ref.export()
        acts = np.array([rng.choice(np.flatnonzero(sc.true_boards(ex)[g].reshape(-1) == 2)) if not ex["done"][g] else -1
                         for g in range(G)], np.int32)
        ref.ply(acts)
    ex = ref.export()
    boards = sc.true_boards(ex)
    cases = []
    for g in range(G):
        if ex["done"][g]:
            continue
        for p in range(6):
            w, cells = playout.playout_winner(boards[g], int(ex["cur"][g]), 5, g, p)
            cases.append((boards[g], int(ex["cur"][g]), w, cells))
    assert cases
    for cur in (0, 1):
        sel = [c for c in cases if c[1] == cur]
        if not sel:
            continue
        replay = hexref.RefBatch(hexref.KIND_GAME_A, N, len(sel))
        replay.set_board(np.stack([c[0] for c in sel]), cur)
        first = np.full(len(sel), -1)
        for k in range(N * N):
            acts = np.array([c[3][k] if k < len(c[3]) else -1 for c in sel], np.int32)
            ret = replay.ply(acts)
            hit = (first < 0) & ((ret == 0) | (ret == 1))
            first[hit] = ret[hit]
        assert np.array_equal(first, [c[2] for c in sel])


@pytest.mark.parametrize("variant,agent_mode,opp_first", sc.ENV_KINDS)
@pytest.mark.parametrize("N", (3, 6, 11, 19))
def test_emulated_env_to_raw_copy_exports_the_source_game(N, variant, agent_mode, opp_first):
    """Env games (WHITE agents transposed) copied into a raw batch: the same regions, exact counters, cur, done and winner;
    then the same plies on the copy and on the reference make_move over the exported state (exact counters) agree."""
    G = 40
    src = env_batch(N, G, 5 + N, variant, agent_mode, opp_first)
    dst = EmuBatch(variant, N, G + 3, raw=True)
    dst.reset()
    before = dst.export()
    rng = np.random.default_rng(N)
    si = rng.permutation(G)
    di = si[::-1].copy()
    copy_games(dst, src, si, di)
    a, b = src.export(), dst.export()
    for k in STATE_KEYS:
        assert np.array_equal(b[k][di], a[k][si]), k
    for k in STATE_KEYS:                                                   # games G, G+1, G+2 were not named
        assert np.array_equal(b[k][G:], before[k][G:]), k
    assert (b["draws"] == 0).all()
    games = [playout.RawGame(b["regions"][g], b["region_counter"][g], b["cur"][g], b["done"][g], b["winner"][g]) for g in range(G + 3)]
    for _ in range(N * N):
        empty = sc.true_boards(b).reshape(G + 3, -1) == 2
        true = np.array([rng.integers(-1, N * N + 1) if rng.uniform() < 0.1 or not empty[g].any() else rng.choice(np.flatnonzero(empty[g]))
                         for g in range(G + 3)], np.int32)
        cur = b["cur"].astype(np.int64)
        acts = true.copy()
        if variant == 1:                                                   # variant B: the mover's view, transposed for WHITE
            ok = (true >= 0) & (true < N * N) & (cur == 1)
            acts[ok] = (true[ok] % N) * N + true[ok] // N
        ret = dst.ply(acts)
        want = np.array([games[g].make_move(int(true[g])) for g in range(G + 3)], np.int8)
        assert np.array_equal(ret, want)
        b = dst.export()
        for g in range(G + 3):
            assert np.array_equal(b["regions"][g], games[g].regions) and list(b["region_counter"][g]) == games[g].counter
            assert b["cur"][g] == games[g].cur and b["winner"][g] == games[g].winner


def test_emulated_copy_broadcast_raw_to_raw_and_out_of_range():
    N, G, C = 7, 6, 5
    src = EmuBatch(1, N, G, raw=True)
    boards, to_move = sc.random_boards(np.random.default_rng(1), G, N)
    src.import_boards(boards, to_move)
    dst = EmuBatch(1, N, G * C + 2, raw=True)
    copy_games(dst, src, np.repeat(np.arange(G), C), None)     # null dst_index: identity
    a, b = src.export(), dst.export()
    for k in STATE_KEYS:
        assert np.array_equal(b[k][:G * C], np.repeat(a[k], C, axis=0)), k
    snap = dst.export()
    copy_games(dst, src, np.array([-1, G, 0, 1]), np.array([0, 1, G * C + 2, -5]))   # every pair out of range
    for k in STATE_KEYS:
        assert np.array_equal(dst.export()[k], snap[k]), k
    copy_games(src, src, np.array([0]), np.array([3]))          # same batch, disjoint sets
    assert np.array_equal(src.export()["regions"][3], a["regions"][0])


def test_abi_argument_checks_without_a_gpu():
    L = _native.lib()
    p = ctypes.c_void_p(8)
    assert L.hexb_copy_games(None, p, None, None, 4, None) == -1
    assert L.hexb_copy_games(p, None, None, None, 4, None) == -1
    assert L.hexb_playouts(None, 32, 0, None, p, None) == -1
    assert L.hexb_version() == (1 << 16) | 5
