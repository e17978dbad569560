"""Shared helpers of the tree-search tests (test_mcts_cpu.py, test_gpu_mcts.py): the tree buffer read through the layout documented
in hex_gym_env_b200/csrc/hexb_mcts.cuh, oracle trees for the roots of a batch, and the whole-tree comparison."""
import numpy as np

from oracle import mcts
import search_common as sc


def parse_tree(buf, N, G):
    """Per root: dict(active, used, s, vsum, to_move, nodes=[dict(flag, nn, child, n, w, p)]) from the raw tree bytes."""
    buf = np.ascontiguousarray(np.asarray(buf, np.uint8))
    C, Cp = N * N, (N * N + 31) // 32 * 32
    head = buf[:128]
    assert int(head[:4].view(np.int32)[0]) == 0x5354434d and int(head[4:8].view(np.int32)[0]) == N
    assert int(head[8:16].view(np.int64)[0]) == G
    max_nodes = int(head[16:20].view(np.int32)[0])
    root_bytes = int(head[40:48].view(np.int64)[0])
    pad = lambda b: (b + 127) // 128 * 128
    off_nn = 128 + pad(8 * N) + pad(8 * (C + 1))
    off_flag = off_nn + pad(4 * max_nodes)
    off_edges = off_flag + pad(4 * max_nodes)
    assert root_bytes == off_edges + 16 * Cp * max_nodes
    roots = []
    for g in range(G):
        r = buf[128 + g * root_bytes:128 + (g + 1) * root_bytes]
        meta = r[:128].view(np.int32)
        used = int(meta[1])
        nn = r[off_nn:off_nn + 4 * max_nodes].view(np.int32)
        flag = r[off_flag:off_flag + 4 * max_nodes].view(np.int32)
        nodes = []
        for k in range(used if meta[0] else 0):
            e = r[off_edges + 16 * Cp * k:off_edges + 16 * Cp * (k + 1)]
            nodes.append(dict(flag=int(flag[k]), nn=int(nn[k]), child=e[:4 * Cp].view(np.int32)[:C],
                              n=e[4 * Cp:8 * Cp].view(np.int32)[:C], w=e[8 * Cp:12 * Cp].view(np.float32)[:C],
                              p=e[12 * Cp:16 * Cp].view(np.float32)[:C]))
        roots.append(dict(active=int(meta[0]), used=used, s=int(meta[2]) & 0xFFFFFFFF, vsum=meta[3:4].view(np.float32)[0],
                          to_move=int(meta[4]), nodes=nodes))
    return roots


def oracle_trees(export, seed, game_offset, variant, max_nodes, c_puct, fpu, first_playout, root_mask=None):
    """One oracle.mcts.RootTree per active root of an exported batch (None for an inactive one)."""
    boards = sc.true_boards(export)
    G = len(export["cur"])
    out = []
    for g in range(G):
        ok = not export["done"][g] and (root_mask is None or root_mask[g])
        out.append(mcts.RootTree(boards[g], int(export["cur"][g]), max_nodes, c_puct, fpu, first_playout, variant, seed,
                                 game_offset + g) if ok else None)
    return out


def same_bits(a, b):
    """Float32 arrays (or scalars) equal bit for bit, except that any NaN matches any NaN: which NaN a sum makes differs between the
    host and the device and is not part of the search's definition (include/hexb.h)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb]))


def assert_trees_equal(roots, oracle):
    """Bit for bit over the whole tree (same_bits for the floats): every node's flag and Nn, every expanded node's edge arrays, the
    root's counters and sum."""
    assert len(roots) == len(oracle)
    for g, (r, o) in enumerate(zip(roots, oracle)):
        if o is None:
            assert r["active"] == 0, g
            continue
        assert r["active"] == 1 and r["to_move"] == o.t0, g
        assert r["used"] == len(o.nodes) and r["s"] == o.s, (g, r["used"], len(o.nodes), r["s"], o.s)
        assert same_bits(r["vsum"], o.vsum), (g, r["vsum"], o.vsum)
        for k, (a, b) in enumerate(zip(r["nodes"], o.nodes)):
            assert a["flag"] == b.flag and a["nn"] == b.nn, (g, k, a["flag"], b.flag, a["nn"], b.nn)
            if b.flag != mcts.EXPANDED:
                continue
            assert np.array_equal(a["child"], b.child), (g, k)
            assert np.array_equal(a["n"], b.n), (g, k)
            assert same_bits(a["w"], b.w), (g, k)
            assert same_bits(a["p"], b.p), (g, k)


def one_move_win_positions(rng, G, N):
    """G random positions (true boards, side to move) where nobody has connected yet and the side to move has a winning cell;
    also the winning cells of each (bool [G, C])."""
    from oracle import playout
    boards, movers, wins = [], [], []
    while len(boards) < G:
        b, t = sc.random_boards(rng, 1, N)
        b, t = b[0], int(t[0])
        if playout.connects(b, 0) or playout.connects(b, 1):
            continue
        w = np.zeros(N * N, bool)
        for c in np.flatnonzero(b.reshape(-1) == 2):
            bb = b.copy().reshape(-1)
            bb[c] = t
            w[c] = playout.connects(bb.reshape(N, N), t)
        if w.any():
            boards.append(b)
            movers.append(t)
            wins.append(w)
    return np.stack(boards), np.array(movers, np.int8), np.stack(wins)


def as_oracle(r):
    """A parsed root in the shape assert_trees_equal expects of an oracle tree (None for an inactive root)."""
    if not r["active"]:
        return None
    o = mcts.RootTree(np.full(1, 2), r["to_move"], 1, 0, 0, 0)
    o.s, o.vsum = r["s"], r["vsum"]
    o.nodes = []
    for nd in r["nodes"]:
        x = mcts.Node(len(nd["n"]), nd["flag"])
        x.nn, x.child, x.n, x.w, x.p = nd["nn"], nd["child"], nd["n"], nd["w"], nd["p"]
        o.nodes.append(x)
    return o


def assert_same_tree(a, b, N, G):
    """Two tree buffers hold the same trees (bytes the layout leaves unused, e.g. free node slots, are not compared)."""
    assert_trees_equal(parse_tree(a, N, G), [as_oracle(r) for r in parse_tree(b, N, G)])


# ---------------------------------------------------------------------------------------------- float edges of the split form
# (test_mcts_edges_cpu.py, test_gpu_mcts_edges.py) c_puct x fpu, and the priors and values expand is handed: zeros of both signs,
# subnormals, numbers near the float32 limit (W overflows to inf), infinities and NaNs of both signs.
EDGE_SETTINGS = [(c, f) for c in (0.0, 1e-30, 1e30, np.inf) for f in (-np.inf, -0.0, np.inf)]
EDGE_PRIORS = np.array([0.0, -0.0, 1e-45, 1e-39, 3e38, -0.5, -3e38, 0.25, 1.0], np.float32)
EDGE_VALUES = np.array([0.0, -0.0, 1.0, -1.0, 3e38, -3e38, np.inf, -np.inf, np.nan, -np.nan], np.float32)


def edge_inputs(rng, G, C):
    """priors f32[G, C] and values f32[G] for one expand: each entry an edge value or, one time in three, an ordinary one."""
    priors = np.where(rng.uniform(size=(G, C)) < 2 / 3, rng.choice(EDGE_PRIORS, size=(G, C)),
                      rng.uniform(0, 1, size=(G, C))).astype(np.float32)
    values = np.where(rng.uniform(size=G) < 2 / 3, rng.choice(EDGE_VALUES, size=G), rng.uniform(-1, 1, size=G)).astype(np.float32)
    return priors, values


def assert_root_outputs_equal(got, want):
    """root() outputs (visits, q, value, nodes_used) of two sides: the counts exactly, the floats by same_bits."""
    visits, q, value, used = (np.asarray(x) for x in got)
    assert np.array_equal(visits, np.asarray(want[0])) and np.array_equal(used, np.asarray(want[3]))
    assert same_bits(q, want[1]) and same_bits(value, want[2])
