"""GPU (-m gpu): the tree-search primitives through libhexb.so - hexb_copy_games against the source games' export and the
reference make_move on the copied state (exact counters), hexb_playouts against the playout oracle bit for bit, both through
torch.ops.hexb and inside a CUDA graph, and the flat Monte-Carlo example against the random opponent."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import playout
import search_common as sc

pytestmark = pytest.mark.gpu

STATE_KEYS = ("regions", "region_counter", "cur", "done", "winner")
ALL_KEYS = ("board", "regions", "region_counter", "cur", "done", "winner", "agent", "draws")


@pytest.fixture(scope="module")
def hb():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import hex_gym_env_b200 as hb
    return hb


def host(ex):
    return {k: v.cpu().numpy() for k, v in ex.items()}


def env_batch(hb, N, G, seed, variant, agent_mode, opponent_first, steps=None, auto_reset=True):
    env = hb.HexBatch(N, G, variant=variant, device=0, seed=seed, agent_mode=agent_mode, opponent_first=opponent_first,
                      auto_reset=auto_reset)
    env.reset()
    for _ in range(sc.env_steps(N) if steps is None else steps):
        env.step(outputs=False)
    return env


def oracle_wins(ex, seed, game_offset, first, P):
    boards = sc.true_boards(ex)
    out = np.full(len(ex["cur"]), -1, np.int32)
    for g in range(len(out)):
        if not ex["done"][g]:
            out[g] = playout.wins(boards[g], int(ex["cur"][g]), seed, game_offset + g, first, P)
    return out


def plies_agree(dst, games, rng, variant, plies):
    """The same hexb_ply actions on the copies and in the reference make_move over their exported state agree ply for ply."""
    N, G = dst.N, dst.G
    b = host(dst.export_state())
    for _ in range(plies):
        empty = sc.true_boards(b).reshape(G, -1) == 2
        true = np.array([rng.integers(-1, N * N + 1) if rng.uniform() < 0.1 or not empty[g].any() else rng.choice(np.flatnonzero(empty[g]))
                         for g in range(G)], np.int32)
        acts = true.copy()
        if variant == 1:                                   # variant B: the mover's view, transposed for WHITE
            ok = (true >= 0) & (true < N * N) & (b["cur"] == 1)
            acts[ok] = (true[ok] % N) * N + true[ok] // N
        ret = dst.ply(torch.from_numpy(acts)).cpu().numpy()
        want = np.array([games[g].make_move(int(true[g])) for g in range(G)], np.int8)
        assert np.array_equal(ret, want)
        b = host(dst.export_state())
        for g in range(G):
            assert np.array_equal(b["regions"][g], games[g].regions) and list(b["region_counter"][g]) == games[g].counter
            assert b["cur"][g] == games[g].cur and b["winner"][g] == games[g].winner


@pytest.mark.parametrize("variant,agent_mode,opp_first", sc.ENV_KINDS)
@pytest.mark.parametrize("N", (3, 7, 11, 19))
def test_copy_env_to_raw(hb, N, variant, agent_mode, opp_first):
    G = 173                                                             # ragged: not a multiple of 32 or 128
    src = env_batch(hb, N, G, 21 + N, variant, agent_mode, opp_first)
    dst = hb.HexBatch(N, G + 40, variant=variant, device=0, raw=True)
    dst.reset()
    boards, to_move = sc.random_boards(np.random.default_rng(N), G + 40, N)
    dst.import_boards(boards, to_move)
    before = host(dst.export_state())
    rng = np.random.default_rng(7 * N + variant)
    si = rng.permutation(G)
    di = rng.permutation(G + 40)[:G]
    dst.copy_games(src, torch.from_numpy(si).cuda(), torch.from_numpy(di).cuda())
    a, b = host(src.export_state()), host(dst.export_state())
    for k in STATE_KEYS:
        assert np.array_equal(b[k][di], a[k][si]), k
    untouched = np.setdiff1d(np.arange(G + 40), di)
    for k in ALL_KEYS:
        assert np.array_equal(b[k][untouched], before[k][untouched]), k
    games = [playout.RawGame(b["regions"][g], b["region_counter"][g], b["cur"][g], b["done"][g], b["winner"][g]) for g in range(G + 40)]
    plies_agree(dst, games, rng, variant, plies=min(N * N, 24))


@pytest.mark.parametrize("variant", (0, 1))
def test_copy_raw_to_raw_identity_broadcast_and_same_handle(hb, variant):
    N, G, C = 9, 50, 7
    src = hb.HexBatch(N, G, variant=variant, device=0, raw=True)
    boards, to_move = sc.random_boards(np.random.default_rng(variant), G, N)
    src.import_boards(boards, to_move)
    a = host(src.export_state())
    ident = hb.HexBatch(N, G, variant=variant, device=0, raw=True)
    ident.copy_games(src)                                               # null indices: the identity over min(G_dst, G_src)
    b = host(ident.export_state())
    for k in STATE_KEYS:
        assert np.array_equal(b[k], a[k]), k
    kids = hb.HexBatch(N, G * C, variant=variant, device=0, raw=True)
    kids.copy_games(src, torch.arange(G, device="cuda").repeat_interleave(C))   # one root into C children
    b = host(kids.export_state())
    for k in STATE_KEYS:
        assert np.array_equal(b[k], np.repeat(a[k], C, axis=0)), k
    snap = host(kids.export_state())
    kids.copy_games(src, torch.tensor([-1, G, 0, 3], device="cuda"), torch.tensor([0, 1, G * C, -2], device="cuda"))
    b = host(kids.export_state())
    for k in ALL_KEYS:                                                  # every pair out of range: nothing written
        assert np.array_equal(b[k], snap[k]), k
    src.copy_games(src, torch.tensor([0, 1], device="cuda"), torch.tensor([10, 11], device="cuda"))   # same handle, disjoint
    b = host(src.export_state())
    for k in STATE_KEYS:
        assert np.array_equal(b[k][[10, 11]], a[k][[0, 1]]), k
        assert np.array_equal(np.delete(b[k], [10, 11], axis=0), np.delete(a[k], [10, 11], axis=0)), k


def test_copy_configuration_mismatches_raise(hb):
    src = hb.HexBatch(7, 16, variant=1, device=0, seed=1, agent_mode=2)
    with pytest.raises(ValueError):
        hb.HexBatch(7, 16, variant=1, device=0, seed=1, agent_mode=2).copy_games(src)       # dst not raw
    with pytest.raises(ValueError):
        hb.HexBatch(8, 16, variant=1, device=0, raw=True).copy_games(src)                   # board size
    with pytest.raises(ValueError):
        hb.HexBatch(7, 16, variant=0, device=0, raw=True).copy_games(src)                   # variant
    dst = hb.HexBatch(7, 16, variant=1, device=0, raw=True)
    with pytest.raises(ValueError):
        dst.copy_games(src, torch.arange(4, device="cuda"), torch.arange(5, device="cuda"))
    from hex_gym_env_b200 import _native
    L = _native.lib()
    other = hb.HexBatch(8, 16, variant=1, device=0, raw=True)
    assert L.hexb_copy_games(other._h, src._h, None, None, 16, None) == -1                  # the C ABI checks it too
    assert L.hexb_copy_games(src._h, dst._h, None, None, 16, None) == -1
    assert L.hexb_copy_games(dst._h, src._h, None, None, -1, None) == -1
    assert L.hexb_playouts(dst._h, 0, 0, None, None, None) == -1


@pytest.mark.parametrize("N", range(3, 20))
def test_playouts_match_the_oracle(hb, N):
    G, P, first = 8, 37, 5
    for variant, agent_mode, opp_first in sc.ENV_KINDS:
        seed = 100 * N + 10 * variant + agent_mode
        env = env_batch(hb, N, G, seed, variant, agent_mode, opp_first)
        w = env.playouts(P, first).cpu().numpy()
        assert np.array_equal(w, oracle_wins(host(env.export_state()), seed, 0, first, P)), (variant, agent_mode)
    rng = np.random.default_rng(N)
    for variant in (0, 1):
        raw = hb.HexBatch(N, G, variant=variant, device=0, seed=2 ** 40 + 9, game_offset=3, raw=True)
        boards, to_move = sc.random_boards(rng, G, N)
        raw.import_boards(boards, to_move)
        w = raw.playouts(P, first).cpu().numpy()
        assert np.array_equal(w, oracle_wins(host(raw.export_state()), 2 ** 40 + 9, 3, first, P)), variant


def test_playouts_of_a_pre_rolled_batch_copied_into_raw(hb):
    """Playouts on the raw copies of env games equal the playouts on the env games (same seed and global indices)."""
    N, G = 11, 300
    env = env_batch(hb, N, G, 5, 1, 2, False)
    raw = hb.HexBatch(N, G, variant=1, device=0, seed=5, raw=True)
    raw.copy_games(env)
    assert torch.equal(env.playouts(64, 3), raw.playouts(64, 3))


def test_playouts_skip_finished_masked_and_unreset_games(hb):
    N, G = 5, 256
    fresh = hb.HexBatch(N, G, variant=1, device=0, seed=3, agent_mode=2)
    assert (fresh.playouts(8) == -1).all()
    env = env_batch(hb, N, G, 3, 1, 2, False, steps=7, auto_reset=False)
    done = env.export_state()["done"].cpu().numpy().astype(bool)
    assert done.any() and not done.all()
    mask = np.ones(G, np.uint8)
    mask[::3] = 0
    w = env.playouts(8, 0, torch.from_numpy(mask)).cpu().numpy()
    assert ((w == -1) == (done | (mask == 0))).all()
    ok = ~done & (mask == 1)
    assert ((w >= 0) & (w <= 8))[ok].all()
    assert np.array_equal(w[ok], env.playouts(8).cpu().numpy()[ok])


def test_torch_ops_and_cuda_graph(hb):
    from hex_gym_env_b200 import torch_ops
    ops = torch_ops.load()
    N, G, C, P = 7, 96, 5, 40
    env = env_batch(hb, N, G, 12, 1, 2, False)
    roots = torch.arange(G, device="cuda").repeat_interleave(C)
    kids_a = hb.HexBatch(N, G * C, variant=1, device=0, seed=12, raw=True)
    kids_b = hb.HexBatch(N, G * C, variant=1, device=0, seed=12, raw=True)
    kids_c = hb.HexBatch(N, G * C, variant=1, device=0, seed=12, raw=True)
    kids_a.copy_games(env, roots)
    want = kids_a.playouts(P, 2)
    ops.copy_games(kids_b.handle, env.handle, roots, None, roots.numel())
    wins_b = torch.empty(G * C, dtype=torch.int32, device="cuda")
    ops.playouts(kids_b.handle, P, 2, None, wins_b)
    assert torch.equal(wins_b, want)
    assert torch.equal(kids_b.export_state()["regions"], kids_a.export_state()["regions"])
    wins_c = torch.full((G * C,), -7, dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        kids_c.copy_games(env, roots)                                  # load the kernels outside the capture
        ops.playouts(kids_c.handle, 1, 0, None, wins_c)
        s.synchronize()
        with torch.cuda.graph(graph, stream=s):
            ops.copy_games(kids_c.handle, env.handle, roots, None, roots.numel())
            ops.playouts(kids_c.handle, P, 2, None, wins_c)
    torch.cuda.current_stream().wait_stream(s)
    wins_c.fill_(-7)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(wins_c, want)
    with pytest.raises(RuntimeError):
        ops.playouts(kids_c.handle, 0, 0, None, wins_c)
    with pytest.raises(RuntimeError):
        ops.copy_games(env.handle, kids_c.handle, None, None, 4)             # dst not raw


# flat Monte-Carlo agent (examples/flat_mc.py) vs the random opponent at 5x5, 1,024 games, 32 playouts per child, 100 env steps:
# deterministic given the seeds. Measured on a B200: 15,520 of 15,528 episodes (0.9995).
FLAT_MC_MIN_WIN_RATE = 0.99


def test_flat_mc_example_beats_the_random_opponent(hb):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    try:
        import flat_mc
    finally:
        sys.path.pop(0)
    r = flat_mc.run(board_size=5, games=1024, playouts=32, steps=100, seed=0)
    print("flat_mc 5x5: agent won %d of %d episodes (%.4f)" % (r["agent_wins"], r["episodes"], r["win_rate"]))
    assert r["episodes"] > 5000 and r["win_rate"] > FLAT_MC_MIN_WIN_RATE
