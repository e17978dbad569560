"""Shared helpers of the tree-reuse tests (test_mcts_advance_cpu.py, test_gpu_mcts_advance.py): hexb_mcts_advance (include/hexb.h)
restated in plain Python and numpy float32 over the oracle's trees (oracle/mcts.py RootTree), and the root positions the tree buffer
holds."""
import numpy as np

from oracle import mcts
import mcts_common as mc
import search_common as sc


def reachable(o, r=0):
    """The nodes of an oracle tree reachable from node r through child pointers (r included), in increasing number."""
    seen, stack = {r}, [r]
    while stack:
        nd = o.nodes[stack.pop()]
        if nd.flag == mcts.EXPANDED:
            for j in nd.child[nd.child >= 0]:
                if int(j) not in seen:
                    seen.add(int(j))
                    stack.append(int(j))
    return sorted(seen)


def advance_path(o, board, to_move):
    """The moves from the root's position to (board, to_move) that advance follows: [] (the same position), [c1] or [c1, c2]
    with c1 the old side to move's stone; None when the new position is not one or two such moves on."""
    b, old, t0, t = np.asarray(board, np.int8).reshape(-1), o.board, o.t0, int(to_move)
    stones = old != mcts.EMPTY
    if (b[stones] != old[stones]).any():
        return None
    added = [int(c) for c in np.flatnonzero(~stones & (b != mcts.EMPTY))]
    if not added and t == t0:
        return []
    if len(added) == 1 and b[added[0]] == t0 and t == t0 ^ 1:
        return added
    if len(added) == 2 and b[added[0]] != b[added[1]] and t == t0:
        return added if b[added[0]] == t0 else added[::-1]
    return None


def advance(o, board, to_move, first_playout):
    """hexb_mcts_advance for one active root (include/hexb.h): the tree re-rooted in place on the node the path reaches, or a
    fresh tree exactly as init leaves it. Returns the root's tree (o itself, or a new RootTree)."""
    b, t = np.array(board, np.int8).reshape(-1), int(to_move)
    path = advance_path(o, b, t)
    node, parent, cell = 0, -1, -1
    if path is not None and o.nodes[0].flag == mcts.EXPANDED:
        for c in path:
            j = int(o.nodes[node].child[c])
            if not (0 <= j < len(o.nodes) and o.nodes[j].flag == mcts.EXPANDED):
                path = None
                break
            parent, cell, node = node, c, j
    else:
        path = None
    if path is None:
        return mcts.RootTree(b, t, o.max_nodes, o.c_puct, o.fpu, first_playout, o.variant, o.seed, o.gid)
    o.leaf, o.first = None, int(first_playout)
    if not path:
        return o
    keep = reachable(o, node)                            # prune: r and its subtree, renumbered in increasing old number
    new = {k: i for i, k in enumerate(keep)}
    edge_n, edge_w = int(o.nodes[parent].n[cell]), o.nodes[parent].w[cell]
    nodes = []
    for k in keep:
        nd = o.nodes[k]
        if nd.flag == mcts.EXPANDED:
            nd.child = np.array([new[int(j)] if j >= 0 else -1 for j in nd.child], np.int32)
        nodes.append(nd)
    o.nodes = nodes
    o.nodes[0].nn = edge_n                               # the root's counters follow the edge into r
    o.s, o.vsum = edge_n, -np.float32(edge_w)
    o.board, o.t0 = b, t
    return o


def oracle_advance(trees, export, seed, game_offset, variant, max_nodes, c_puct, fpu, first_playout, root_mask=None, live=None):
    """hexb_mcts_advance over the oracle trees of a batch (None = inactive) after its games moved on to `export`. live: the games
    ever reset (an export does not show it), None = all."""
    boards = sc.true_boards(export)
    out = []
    for g, o in enumerate(trees):
        ok = not export["done"][g] and (root_mask is None or root_mask[g]) and (live is None or live[g])
        if not ok:
            out.append(None)
        elif o is None:
            out.append(mcts.RootTree(boards[g], int(export["cur"][g]), max_nodes, c_puct, fpu, first_playout, variant, seed,
                                     game_offset + g))
        else:
            out.append(advance(o, boards[g], int(export["cur"][g]), first_playout))
    return out


def root_boards(buf, N, G):
    """Each root's position from its rows in the tree buffer: true boards i8[G, C] (0 BLACK, 1 WHITE, 2 EMPTY)."""
    buf = np.ascontiguousarray(np.asarray(buf, np.uint8))
    root_bytes = int(buf[40:48].view(np.int64)[0])
    out = np.full((G, N * N), 2, np.int8)
    for g in range(G):
        rows = buf[128 + g * root_bytes + 128:128 + g * root_bytes + 128 + 8 * N].view(np.uint32)
        for y in range(N):
            for x in range(N):
                if not (rows[N + y] >> x) & 1:
                    out[g, y * N + x] = 0 if (rows[y] >> x) & 1 else 1
    return out


def assert_advanced_trees_equal(buf, N, G, oracle):
    """mcts_common.assert_trees_equal, and every active root's position equals the oracle's."""
    mc.assert_trees_equal(mc.parse_tree(buf, N, G), oracle)
    boards = root_boards(buf, N, G)
    for g, o in enumerate(oracle):
        if o is not None:
            assert np.array_equal(boards[g], o.board), g
