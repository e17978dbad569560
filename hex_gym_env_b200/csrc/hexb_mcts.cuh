// hexb_mcts.cuh - batched Monte-Carlo tree search (PUCT), one tree per game of a handle. The search itself is defined in
// include/hexb.h; this file holds the per-root pieces the kernels of hexb_step_inst.cu are made of. A root is searched by one
// warp: lane l owns cells l, l + 32, ... of every node and path entries l, l + 32, ...; the warp-wide steps are the mc_* helpers
// below. Compiled for the host (tests/emu, HEXB_HOST_EMU) the "warp" is one lane that owns every cell and every entry, so the
// emulator runs this same source with loops in place of the shuffles.
//
// Tree buffer layout (hexb_mcts_tree_bytes). Every section is a multiple of 128 bytes; Cp = C rounded up to a multiple of 32.
//   [0, 128)                       header, byte offsets: 0 i32 magic 'MCTS', 4 i32 N, 8 i64 G, 16 i32 max_nodes, 20 f32 c_puct,
//                                  24 f32 fpu, 32 i64 first_playout, 40 i64 root_bytes
//   128 + g * root_bytes           root g:
//     + 0                          meta i32[32]: [0] active, [1] nodes used, [2] simulations done s (u32), [3] value sum (f32 bits,
//                                  from the root's side to move), [4] root's true colour to move, [5] pending (split form),
//                                  [6] depth D of the pending leaf, [7] its node (-1 = a new position), [8] its parent node,
//                                  [9] the cell into it (true row-major)
//     + 128                        root rows u32[2N]: black[0..N), empty[0..N) in true orientation (bit x of row y = cell (y, x))
//     + off_path                   path i32[2 (C + 1)]: node[0..C] (-1 = leaf not stored), cell[0..C] (cell[d]: the move into depth d)
//     + off_nn                     Nn i32[max_nodes]: simulations whose path contained the node
//     + off_flag                   flag i32[max_nodes]: 0 unexpanded (node 0 before its first simulation), 1 expanded, 2 terminal
//     + off_edges + n * 16 Cp      node n's edges, structure of arrays over the true row-major cell c < Cp:
//                                  child i32[Cp] (-1 = none), N i32[Cp], W f32[Cp], P f32[Cp] (0 for cells not empty at the node)
// Edge arrays are written only when a node is expanded; a terminal node has none.
// Within one advance launch (mc_advance_root) a flag word also carries scratch: bit 2 marks a node of the kept subtree and bits
// 3.. hold its new number. Every flag word is 0, 1 or 2 again when the launch ends.
#pragma once
#include <math.h>
#include <string.h>

#include "hexb_search.cuh"

namespace hexb {

constexpr int32_t kMctsMagic = 0x5354434d;      // 'MCTS'
constexpr int kMctsMaxNodes = 1 << 24;          // visit counts stay exact in float32
constexpr int kMctsMaxPlayouts = 1 << 16;
enum : int { MF_UNEXPANDED = 0, MF_EXPANDED = 1, MF_TERMINAL = 2 };
enum : int { MM_ACTIVE = 0, MM_USED, MM_SIMS, MM_VSUM, MM_TOMOVE, MM_PENDING, MM_DEPTH, MM_NODE, MM_PARENT, MM_CELL };

HEXB_HD long long mc_pad128(long long b) { return (b + 127) & ~127ll; }
HEXB_HD int mc_cp(int N) { return (N * N + 31) & ~31; }
HEXB_HD long long mc_off_path(int N) { return 128 + mc_pad128(8ll * N); }
HEXB_HD long long mc_off_nn(int N) { return mc_off_path(N) + mc_pad128(8ll * (N * N + 1)); }
HEXB_HD long long mc_off_flag(int N, int max_nodes) { return mc_off_nn(N) + mc_pad128(4ll * max_nodes); }
HEXB_HD long long mc_off_edges(int N, int max_nodes) { return mc_off_flag(N, max_nodes) + mc_pad128(4ll * max_nodes); }
HEXB_HD long long mc_root_bytes(int N, int max_nodes) { return mc_off_edges(N, max_nodes) + 16ll * mc_cp(N) * max_nodes; }

// ---------------------------------------------------------------------------------------------- the warp
#if defined(__CUDA_ARCH__)
HEXB_HD int mc_lane() { return threadIdx.x & 31; }
HEXB_HD int mc_width() { return 32; }
HEXB_HD unsigned long long mc_max(unsigned long long k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long x = __shfl_xor_sync(0xffffffffu, k, o);
        k = x > k ? x : k;
    }
    return k;
}
HEXB_HD int mc_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }
// the lanes below this one with p set; total: the lanes with p set
HEXB_HD int mc_prefix(bool p, int &total) {
    const unsigned b = __ballot_sync(0xffffffffu, p);
    total = __popc(b);
    return __popc(b & ((1u << (threadIdx.x & 31)) - 1u));
}
HEXB_HD void mc_sync() { __syncwarp(); }
// float32 arithmetic rounded once per operation, never contracted into an FMA (numpy float32 reproduces it)
HEXB_HD float f_mul(float a, float b) { return __fmul_rn(a, b); }
HEXB_HD float f_div(float a, float b) { return __fdiv_rn(a, b); }
HEXB_HD float f_add(float a, float b) { return __fadd_rn(a, b); }
HEXB_HD float f_sqrt(float a) { return __fsqrt_rn(a); }
HEXB_HD uint32_t f_bits(float f) { return __float_as_uint(f); }
HEXB_HD float bits_f(uint32_t u) { return __uint_as_float(u); }
#else
HEXB_HD int mc_lane() { return 0; }
HEXB_HD int mc_width() { return 1; }
HEXB_HD unsigned long long mc_max(unsigned long long k) { return k; }
HEXB_HD int mc_sum(int v) { return v; }
HEXB_HD int mc_prefix(bool p, int &total) {
    total = p ? 1 : 0;
    return 0;
}
HEXB_HD void mc_sync() {}
HEXB_HD float f_mul(float a, float b) { return a * b; }   // SSE: one rounding per operation (no FMA on the baseline x86-64 target)
HEXB_HD float f_div(float a, float b) { return a / b; }
HEXB_HD float f_add(float a, float b) { return a + b; }
HEXB_HD float f_sqrt(float a) { return sqrtf(a); }
HEXB_HD uint32_t f_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
HEXB_HD float bits_f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
#endif

// ---------------------------------------------------------------------------------------------- the tree
struct MctsArgs {
    uint8_t *tree;
    unsigned long long tree_bytes;
    unsigned long long seed, game_offset;
    int max_nodes;                 // init
    float c_puct, fpu;             // init
    long long first_playout;       // init, advance
    const uint8_t *root_mask;      // init, advance: [G] nullable
    int sims, playouts;            // search
    void *leaf_obs;                // select: obs dtype [G, C]
    uint8_t *leaf_mask, *pending;  // select: [G, C], [G]
    const float *priors, *values;  // expand: [G, C], [G]
    int32_t *visits, *nodes_used;  // root: [G, C], [G] (nullable)
    float *q, *value;              // root: [G, C], [G] (nullable)
};

struct Tree {
    uint8_t *base;
    long long G, root_bytes, off_path, off_nn, off_flag, off_edges;
    int N, C, Cp, max_nodes;
    float c_puct, fpu;
    long long first;
};

HEXB_HD void mc_layout(Tree &T, int N, long long G, int max_nodes) {
    T.N = N;
    T.C = N * N;
    T.Cp = mc_cp(N);
    T.G = G;
    T.max_nodes = max_nodes;
    T.root_bytes = mc_root_bytes(N, max_nodes);
    T.off_path = mc_off_path(N);
    T.off_nn = mc_off_nn(N);
    T.off_flag = mc_off_flag(N, max_nodes);
    T.off_edges = mc_off_edges(N, max_nodes);
}

// The tree a search / select / expand / root call works on, from the header init wrote. false: the buffer holds no tree of this
// handle (never initialised, another board size or batch, or smaller than the tree): the call writes nothing.
HEXB_HD bool mc_tree(const MctsArgs &A, int N, long long G, Tree &T) {
    if (!A.tree || A.tree_bytes < 128) return false;
    const int32_t *h = reinterpret_cast<const int32_t *>(A.tree);
    const long long hG = *reinterpret_cast<const long long *>(A.tree + 8);
    const int mn = h[4];
    if (h[0] != kMctsMagic || h[1] != N || hG != G || mn < 1 || mn > kMctsMaxNodes) return false;
    mc_layout(T, N, G, mn);
    if (*reinterpret_cast<const long long *>(A.tree + 40) != T.root_bytes) return false;
    if ((unsigned long long)T.root_bytes * (unsigned long long)G + 128ull > A.tree_bytes) return false;
    T.base = A.tree;
    T.c_puct = bits_f((uint32_t)h[5]);
    T.fpu = bits_f((uint32_t)h[6]);
    T.first = *reinterpret_cast<const long long *>(A.tree + 32);
    return true;
}

HEXB_HD uint8_t *mc_root(const Tree &T, long long g) { return T.base + 128 + g * T.root_bytes; }
HEXB_HD int32_t *mc_meta(const Tree &T, long long g) { return reinterpret_cast<int32_t *>(mc_root(T, g)); }
HEXB_HD uint32_t *mc_rows(const Tree &T, long long g) { return reinterpret_cast<uint32_t *>(mc_root(T, g) + 128); }
HEXB_HD int32_t *mc_path_node(const Tree &T, long long g) { return reinterpret_cast<int32_t *>(mc_root(T, g) + T.off_path); }
HEXB_HD int32_t *mc_path_cell(const Tree &T, long long g) { return mc_path_node(T, g) + T.C + 1; }
HEXB_HD int32_t *mc_nn(const Tree &T, long long g) { return reinterpret_cast<int32_t *>(mc_root(T, g) + T.off_nn); }
HEXB_HD int32_t *mc_flag(const Tree &T, long long g) { return reinterpret_cast<int32_t *>(mc_root(T, g) + T.off_flag); }
HEXB_HD int32_t *mc_child(const Tree &T, long long g, int n) {
    return reinterpret_cast<int32_t *>(mc_root(T, g) + T.off_edges + 16ll * T.Cp * n);
}
HEXB_HD int32_t *mc_edge_n(const Tree &T, long long g, int n) { return mc_child(T, g, n) + T.Cp; }
HEXB_HD float *mc_edge_w(const Tree &T, long long g, int n) { return reinterpret_cast<float *>(mc_child(T, g, n) + 2 * T.Cp); }
HEXB_HD float *mc_edge_p(const Tree &T, long long g, int n) { return reinterpret_cast<float *>(mc_child(T, g, n) + 3 * T.Cp); }

// init's header (written once per launch)
HEXB_HD void mc_write_header(const MctsArgs &A, int N, long long G) {
    int32_t *h = reinterpret_cast<int32_t *>(A.tree);
    h[0] = kMctsMagic;
    h[1] = N;
    *reinterpret_cast<long long *>(A.tree + 8) = G;
    h[4] = A.max_nodes;
    h[5] = (int32_t)f_bits(A.c_puct);
    h[6] = (int32_t)f_bits(A.fpu);
    h[7] = 0;
    *reinterpret_cast<long long *>(A.tree + 32) = A.first_playout;
    *reinterpret_cast<long long *>(A.tree + 40) = mc_root_bytes(N, A.max_nodes);
}

// ---------------------------------------------------------------------------------------------- positions
// Rows are only ever indexed by unrolled compare-and-select, so that they stay in registers.
template <int N>
HEXB_HD uint32_t row_bit(const uint32_t (&rows)[N], int c) {
    const int y = c / N, x = c - y * N;
    uint32_t r = 0u;
#pragma unroll
    for (int yy = 0; yy < N; ++yy) r |= yy == y ? rows[yy] : 0u;
    return (r >> x) & 1u;
}

template <int N>
HEXB_HD void mc_play(uint32_t (&black)[N], uint32_t (&empty)[N], int c, int colour) {
    const int y = c / N;
    const uint32_t bit = 1u << (c - y * N);
#pragma unroll
    for (int yy = 0; yy < N; ++yy) {
        const uint32_t m = yy == y ? bit : 0u;
        empty[yy] &= ~m;
        black[yy] |= colour == 0 ? m : 0u;
    }
}

template <int N>
HEXB_HD void mc_load_root(const Tree &T, long long g, uint32_t (&black)[N], uint32_t (&empty)[N]) {
    const uint32_t *r = mc_rows(T, g);
#pragma unroll
    for (int y = 0; y < N; ++y) {
        black[y] = r[y];
        empty[y] = r[N + y];
    }
}

// Does `colour` connect its edges? WHITE is tested as BLACK on the transposed rows (the neighbourhood is symmetric under it).
template <int N>
HEXB_HD bool mc_connects(const uint32_t (&black)[N], const uint32_t (&empty)[N], int colour) {
    if (colour == 0) return black_connects<N>(black);
    uint32_t t[N];
#pragma unroll
    for (int x = 0; x < N; ++x) {
        uint32_t col = 0u;
#pragma unroll
        for (int y = 0; y < N; ++y) col |= ((~(black[y] | empty[y]) >> x) & 1u) << y;
        t[x] = col;
    }
    return black_connects<N>(t);
}

template <int N>
HEXB_HD int mc_empties(const uint32_t (&empty)[N]) {
    int n = 0;
#pragma unroll
    for (int y = 0; y < N; ++y) n += popc32(empty[y]);
    return n;
}

// the per-cell index of true cell c for the side to move `colour`: hexb_ply's action of a raw handle of this variant
HEXB_HD int mc_action(int variant, int colour, int N, int c) {
    if (variant != VARIANT_B || colour == 0) return c;
    const int y = c / N;
    return (c - y * N) * N + y;
}

// ---------------------------------------------------------------------------------------------- one simulation
// PUCT key of every empty cell of an expanded node; the largest wins. Score bits made order-preserving as unsigned, in the high
// half; 0xffffffff - cell in the low half breaks ties towards the lowest cell. 0 = no empty cell.
template <int N>
HEXB_HD int mc_best_cell(const Tree &T, long long g, int node, const uint32_t (&empty)[N]) {
    const int32_t *en = mc_edge_n(T, g, node);
    const float *ew = mc_edge_w(T, g, node), *ep = mc_edge_p(T, g, node);
    const float sq = f_sqrt((float)mc_nn(T, g)[node]);
    unsigned long long best = 0ull;
    for (int c = mc_lane(); c < T.C; c += mc_width()) {
        if (!row_bit<N>(empty, c)) continue;
        const int n = en[c];
        const float q = n > 0 ? f_div(ew[c], (float)n) : T.fpu;
        const float u = f_div(f_mul(f_mul(T.c_puct, ep[c]), sq), (float)(1 + n));
        const uint32_t b = f_bits(f_add(q, u));
        const uint32_t ord = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
        const unsigned long long key = ((unsigned long long)ord << 32) | (0xffffffffu - (uint32_t)c);
        best = key > best ? key : best;
    }
    best = mc_max(best);
    return best ? (int)(0xffffffffu - (uint32_t)best) : -1;
}

struct MctsLeaf {
    int depth;   // D: path nodes 0..D, moves 1..D
    int node;    // the leaf's node, -1 = a position not in the tree
    int parent;  // node at depth D - 1 (D >= 1)
    int cell;    // the move into the leaf (D >= 1)
};

// Step 1 from node 0: rows end at the leaf's position; path entries are written by their owner lanes.
template <int N>
HEXB_HD MctsLeaf mc_descend(const Tree &T, long long g, int used, int to_move, uint32_t (&black)[N], uint32_t (&empty)[N]) {
    const int lane = mc_lane(), width = mc_width();
    int32_t *pn = mc_path_node(T, g), *pc = mc_path_cell(T, g);
    const int32_t *flag = mc_flag(T, g);
    MctsLeaf L;
    L.depth = 0;
    L.node = 0;
    L.parent = -1;
    L.cell = -1;
    if (lane == 0) pn[0] = 0;
    while (L.depth < T.C && flag[L.node] == MF_EXPANDED) {
        const int c = mc_best_cell<N>(T, g, L.node, empty);
        if (c < 0) break;   // no empty cell left: the node itself is evaluated again
        mc_play<N>(black, empty, c, to_move ^ (L.depth & 1));
        const int child = mc_child(T, g, L.node)[c];
        L.parent = L.node;
        L.cell = c;
        L.node = child >= 0 && child < used ? child : -1;
        ++L.depth;
        if (L.depth % width == lane) {
            pn[L.depth] = L.node;
            pc[L.depth] = c;
        }
        if (L.node < 0 || flag[L.node] == MF_TERMINAL) break;
    }
    return L;
}

// Step 3: the leaf becomes a node (expanded with priors, or terminal) if it is not one yet and the pool has room; node 0 is
// expanded in place at its first simulation. pri: the leaf's priors in its mover's action order (null = 1 / n_empty). Returns
// the number of nodes used.
template <int N>
HEXB_HD int mc_store(const Tree &T, long long g, const MctsLeaf &L, int used, bool terminal, const uint32_t (&empty)[N], int colour,
                     int variant, const float *pri) {
    int n = L.node;
    const bool stored = n >= 0 && mc_flag(T, g)[n] != MF_UNEXPANDED;
    mc_sync();   // every lane has read the flags of this simulation (mc_descend, the line above) before lane 0 writes one
    if (n >= 0) {
        if (stored) return used;
    } else {
        if (used >= T.max_nodes) return used;
        n = used++;
        if (L.depth % mc_width() == mc_lane()) mc_path_node(T, g)[L.depth] = n;   // the entry's owner wrote it in mc_descend
        if (mc_lane() == 0) {
            mc_child(T, g, L.parent)[L.cell] = n;
            mc_nn(T, g)[n] = 0;
        }
    }
    if (mc_lane() == 0) mc_flag(T, g)[n] = terminal ? MF_TERMINAL : MF_EXPANDED;
    if (terminal) return used;
    const float uni = pri ? 0.0f : f_div(1.0f, (float)mc_empties<N>(empty));
    int32_t *ch = mc_child(T, g, n), *en = mc_edge_n(T, g, n);
    float *ew = mc_edge_w(T, g, n), *ep = mc_edge_p(T, g, n);
    for (int c = mc_lane(); c < T.Cp; c += mc_width()) {
        const bool e = c < T.C && row_bit<N>(empty, c);
        ch[c] = -1;
        en[c] = 0;
        ew[c] = 0.0f;
        ep[c] = !e ? 0.0f : (pri ? pri[mc_action(variant, colour, N, c)] : uni);
    }
    return used;
}

// Step 4 for path entries 0..D (after an mc_sync: the entries were written by other lanes). v: the leaf's value for its side
// to move; the edge into depth d gets it for the player who made that move.
HEXB_HD void mc_backup(const Tree &T, long long g, int D, int used, float v) {
    const int32_t *pn = mc_path_node(T, g), *pc = mc_path_cell(T, g);
    int32_t *nn = mc_nn(T, g);
    for (int d = mc_lane(); d <= D; d += mc_width()) {
        const int n = pn[d];
        if (n >= 0 && n < used) nn[n] += 1;
        if (d == 0) continue;
        const int p = pn[d - 1], c = pc[d];
        if (p < 0 || p >= used || c < 0 || c >= T.C) continue;
        mc_edge_n(T, g, p)[c] += 1;
        float *w = mc_edge_w(T, g, p) + c;
        *w = f_add(*w, ((D - d) & 1) ? v : -v);
    }
}

// ---------------------------------------------------------------------------------------------- per-root calls
// init's state of root g (one thread): node 0 unexpanded on (black, empty) with true colour to_move to move; -1 = inactive
template <int N>
HEXB_HD void mc_fresh_root(const Tree &T, long long g, int to_move, const uint32_t (&black)[N], const uint32_t (&empty)[N]) {
    int32_t *m = mc_meta(T, g);
    for (int i = 0; i < 32; ++i) m[i] = 0;
    m[MM_NODE] = -1;
    if (to_move < 0) return;
    m[MM_ACTIVE] = 1;
    m[MM_USED] = 1;
    m[MM_TOMOVE] = to_move;
    uint32_t *r = mc_rows(T, g);
#pragma unroll
    for (int y = 0; y < N; ++y) {
        r[y] = black[y];
        r[N + y] = empty[y];
    }
    mc_nn(T, g)[0] = 0;
    mc_flag(T, g)[0] = MF_UNEXPANDED;
}

// init: one thread per root
template <int N>
HEXB_HD void mc_init_root(const View &V, const MctsArgs &A, long long g) {
    Tree T;
    mc_layout(T, N, V.G, A.max_nodes);
    T.base = A.tree;
    uint32_t black[N], empty[N];
    const int to_move = (A.root_mask && !A.root_mask[g]) ? -1 : playout_rows<N>(V, g, black, empty);
    mc_fresh_root<N>(T, g, to_move, black, empty);
}

// fused form: all simulations of one root (one warp)
template <int N>
HEXB_HD void mc_search_root(const Tree &T, const MctsArgs &A, int variant, long long g) {
    int32_t *m = mc_meta(T, g);
    if (!m[MM_ACTIVE]) return;
    const int t0 = m[MM_TOMOVE] & 1, P = A.playouts;
    int used = m[MM_USED] < 1 ? 1 : (m[MM_USED] > T.max_nodes ? T.max_nodes : m[MM_USED]);
    uint32_t s = (uint32_t)m[MM_SIMS];
    float vsum = bits_f((uint32_t)m[MM_VSUM]);
    const unsigned long long gid = A.game_offset + (unsigned long long)g;
    for (int it = 0; it < A.sims; ++it) {
        uint32_t black[N], empty[N];
        mc_load_root<N>(T, g, black, empty);
        const MctsLeaf L = mc_descend<N>(T, g, used, t0, black, empty);
        const int mover = t0 ^ (L.depth & 1);
        float v = -1.0f;
        bool terminal = L.node >= 0 && mc_flag(T, g)[L.node] == MF_TERMINAL;
        if (!terminal && L.node < 0) terminal = mc_connects<N>(black, empty, mover ^ 1);
        if (!terminal) {
            const uint32_t p0 = (uint32_t)T.first + s * (uint32_t)P;
            int won = 0;
            for (int j = mc_lane(); j < P; j += mc_width())
                won += playout_winner<N>(black, empty, mover, A.seed, gid, p0 + (uint32_t)j) == mover;
            won = mc_sum(won);
            v = f_div((float)(2 * won - P), (float)P);
        }
        if (!(terminal && L.node >= 0)) used = mc_store<N>(T, g, L, used, terminal, empty, mover, variant, nullptr);
        mc_sync();
        mc_backup(T, g, L.depth, used, v);
        mc_sync();
        vsum = f_add(vsum, (L.depth & 1) ? -v : v);
        ++s;
    }
    if (mc_lane() == 0) {
        m[MM_USED] = used;
        m[MM_SIMS] = (int32_t)s;
        m[MM_VSUM] = (int32_t)f_bits(vsum);
    }
}

// split form, step 1 (one warp per root): a leaf that needs the caller's evaluation is written to leaf_obs / leaf_mask as
// hexb_encode(view 1) of a raw game holding it; a terminal leaf is backed up here.
template <int N>
HEXB_HD void mc_select_root(const Tree &T, const View &V, const MctsArgs &A, long long g) {
    int32_t *m = mc_meta(T, g);
    const bool lead = mc_lane() == 0;
    if (!m[MM_ACTIVE]) {
        if (lead) A.pending[g] = 0;
        return;
    }
    const int t0 = m[MM_TOMOVE] & 1;
    int used = m[MM_USED] < 1 ? 1 : (m[MM_USED] > T.max_nodes ? T.max_nodes : m[MM_USED]);
    uint32_t black[N], empty[N];
    mc_load_root<N>(T, g, black, empty);
    const MctsLeaf L = mc_descend<N>(T, g, used, t0, black, empty);
    const int mover = t0 ^ (L.depth & 1);
    bool terminal = L.node >= 0 && mc_flag(T, g)[L.node] == MF_TERMINAL;
    if (!terminal && L.node < 0) terminal = mc_connects<N>(black, empty, mover ^ 1);
    if (terminal) {
        if (L.node < 0) used = mc_store<N>(T, g, L, used, true, empty, mover, V.variant, nullptr);
        mc_sync();
        mc_backup(T, g, L.depth, used, -1.0f);
        mc_sync();
        if (lead) {
            m[MM_USED] = used;
            m[MM_SIMS] += 1;
            m[MM_VSUM] = (int32_t)f_bits(f_add(bits_f((uint32_t)m[MM_VSUM]), (L.depth & 1) ? 1.0f : -1.0f));
            m[MM_PENDING] = 0;
            A.pending[g] = 0;
        }
        return;
    }
    const int C = N * N;
    const bool opp = V.variant == VARIANT_B && mover == 1;
    for (int c = mc_lane(); c < C; c += mc_width()) {
        const int a = mc_action(V.variant, mover, N, c);
        const uint32_t b = row_bit<N>(empty, c) ? 0u : (row_bit<N>(black, c) ? 0x01u : 0x81u);   // a raw game's label byte
        uint32_t mk;
        const uint32_t ob = encode_byte(b, V.variant, opp, mk);
        store_obs(reinterpret_cast<int8_t *>(A.leaf_obs), V.obs_f32, g * C + a, ob);
        A.leaf_mask[g * C + a] = (uint8_t)mk;
    }
    if (lead) {
        m[MM_PENDING] = 1;
        m[MM_DEPTH] = L.depth;
        m[MM_NODE] = L.node;
        m[MM_PARENT] = L.parent;
        m[MM_CELL] = L.cell;
        A.pending[g] = 1;
    }
}

// split form, steps 2-4 for a pending root (one warp per root): the position is replayed from the stored path
template <int N>
HEXB_HD void mc_expand_root(const Tree &T, const View &V, const MctsArgs &A, long long g) {
    int32_t *m = mc_meta(T, g);
    if (!m[MM_ACTIVE] || !m[MM_PENDING]) return;
    mc_sync();   // every lane has read the flag before it is cleared
    if (mc_lane() == 0) m[MM_PENDING] = 0;
    const int t0 = m[MM_TOMOVE] & 1;
    int used = m[MM_USED] < 1 ? 1 : (m[MM_USED] > T.max_nodes ? T.max_nodes : m[MM_USED]);
    MctsLeaf L;
    L.depth = m[MM_DEPTH];
    L.node = m[MM_NODE];
    L.parent = m[MM_PARENT];
    L.cell = m[MM_CELL];
    if (L.depth < 0 || L.depth > T.C || L.node < -1 || L.node >= used) return;
    if (L.depth == 0 ? L.node != 0 : (L.parent < 0 || L.parent >= used || L.cell < 0 || L.cell >= T.C)) return;
    uint32_t black[N], empty[N];
    mc_load_root<N>(T, g, black, empty);
    const int32_t *pc = mc_path_cell(T, g);
    for (int d = 1; d <= L.depth; ++d) mc_play<N>(black, empty, pc[d], t0 ^ ((d - 1) & 1));   // written by the select launch
    const int mover = t0 ^ (L.depth & 1);
    const float v = A.values[g];
    used = mc_store<N>(T, g, L, used, false, empty, mover, V.variant, A.priors + g * (long long)T.C);
    mc_sync();
    mc_backup(T, g, L.depth, used, v);
    mc_sync();
    if (mc_lane() == 0) {
        m[MM_USED] = used;
        m[MM_SIMS] += 1;
        m[MM_VSUM] = (int32_t)f_bits(f_add(bits_f((uint32_t)m[MM_VSUM]), (L.depth & 1) ? -v : v));
    }
}

// the root's edges in its mover's action order, value sum / Nn, nodes used (0 for an inactive root) - one warp per root
HEXB_HD void mc_root_out(const Tree &T, int variant, const MctsArgs &A, long long g) {
    const int32_t *m = mc_meta(T, g);
    const int C = T.C, N = T.N;
    const bool on = m[MM_ACTIVE] != 0;
    const bool edges = on && mc_flag(T, g)[0] == MF_EXPANDED;
    const int colour = m[MM_TOMOVE] & 1;
    const int32_t *en = mc_edge_n(T, g, 0);
    const float *ew = mc_edge_w(T, g, 0);
    for (int c = mc_lane(); c < C; c += mc_width()) {
        const long long i = g * C + mc_action(variant, colour, N, c);
        const int n = edges ? en[c] : 0;
        if (A.visits) A.visits[i] = n;
        if (A.q) A.q[i] = n > 0 ? f_div(ew[c], (float)n) : 0.0f;
    }
    if (mc_lane() == 0) {
        const int nn = on ? mc_nn(T, g)[0] : 0;
        if (A.value) A.value[g] = nn > 0 ? f_div(bits_f((uint32_t)m[MM_VSUM]), (float)nn) : 0.0f;
        if (A.nodes_used) A.nodes_used[g] = on ? m[MM_USED] : 0;
    }
}

// advance's header field (written once per launch; no per-root code of that launch reads it)
HEXB_HD void mc_write_first_playout(const MctsArgs &A) { *reinterpret_cast<long long *>(A.tree + 32) = A.first_playout; }

// advance (one warp per root): keep the subtree under the game's current position, or start a fresh tree as init does
template <int N>
HEXB_HD void mc_advance_root(const Tree &T, const View &V, const MctsArgs &A, long long g) {
    int32_t *m = mc_meta(T, g);
    const int lane = mc_lane(), width = mc_width();
    const bool lead = lane == 0;
    uint32_t black[N], empty[N];
    const int tn = (A.root_mask && !A.root_mask[g]) ? -1 : playout_rows<N>(V, g, black, empty);
    // the moves from the old root's position P to the new one P': k = 0, 1 or 2 (c1 by the old side to move), -1 = no path
    int k = -1, c1 = -1, c2 = -1;
    if (tn >= 0 && m[MM_ACTIVE]) {
        const int t0 = m[MM_TOMOVE] & 1;
        const uint32_t *rows = mc_rows(T, g);
        bool same = true;
        int nb = 0, nw = 0, cb = -1, cw = -1;
#pragma unroll
        for (int y = 0; y < N; ++y) {
            const uint32_t ob = rows[y], oe = rows[N + y], stones = ~oe & ((1u << N) - 1u);
            same = same && (stones & empty[y]) == 0u && ((ob ^ black[y]) & stones) == 0u;   // every stone of P stays, same colour
            const uint32_t add = oe & ~empty[y], ab = add & black[y], aw = add & ~black[y];
            nb += popc32(ab);
            nw += popc32(aw);
            if (ab) cb = y * N + nth_set_bit(ab, 0);
            if (aw) cw = y * N + nth_set_bit(aw, 0);
        }
        const int mine = t0 == 0 ? nb : nw, c_mine = t0 == 0 ? cb : cw, c_other = t0 == 0 ? cw : cb;
        if (same && nb + nw == 0 && tn == t0) {
            k = 0;
        } else if (same && nb + nw == 1 && mine == 1 && tn == (t0 ^ 1)) {
            k = 1;
            c1 = c_mine;
        } else if (same && nb == 1 && nw == 1 && tn == t0) {
            k = 2;
            c1 = c_mine;
            c2 = c_other;
        }
    }
    // walk the path from node 0: every node on it, and the node r reached, expanded; every child on it stored
    const int used = m[MM_USED] < 1 ? 1 : (m[MM_USED] > T.max_nodes ? T.max_nodes : m[MM_USED]);
    int32_t *fl = mc_flag(T, g);
    int r = 0, parent = -1, cell = -1;
    if (k >= 0 && fl[0] != MF_EXPANDED) k = -1;
    for (int d = 0; d < k; ++d) {
        const int c = d == 0 ? c1 : c2, j = mc_child(T, g, r)[c];
        if (j < 0 || j >= used || fl[j] != MF_EXPANDED) {
            k = -1;
            break;
        }
        parent = r;
        cell = c;
        r = j;
    }
    if (k < 0) {
        mc_sync();   // every lane has read the meta and the flags before lane 0 rewrites them
        if (lead) mc_fresh_root<N>(T, g, tn, black, empty);
        return;
    }
    int kept = used;
    if (k > 0) {
        const int32_t en = mc_edge_n(T, g, parent)[cell];   // the edge into r (its parent's slot is reused below)
        const float ew = mc_edge_w(T, g, parent)[cell];
        int32_t *nn = mc_nn(T, g);
        // 1 mark r and every node reachable from it: a node is numbered after its parent, so one ascending pass sees a node's
        //   mark before it reaches the node's children
        mc_sync();
        if (lead) fl[r] |= 4;
        mc_sync();
        for (int n = r; n < used; ++n) {
            if (fl[n] == (4 | MF_EXPANDED)) {
                const int32_t *ch = mc_child(T, g, n);
                for (int c = lane; c < T.C; c += width) {
                    const int j = ch[c];
                    if (j >= 0 && j < used) fl[j] |= 4;
                }
            }
            mc_sync();
        }
        // 2 new numbers in increasing old number (bits 3..)
        kept = 0;
        for (int base = r; base < used; base += width) {
            const int n = base + lane;
            const int f = n < used ? fl[n] : 0;
            int total;
            const int before = mc_prefix((f & 4) != 0, total);
            if (f & 4) fl[n] = (f & 7) | ((kept + before) << 3);
            kept += total;
        }
        mc_sync();
        // 3 move node n to its new number m <= n with its children renumbered: a child j > n has not moved yet, so its slot still
        //   holds its new number; every slot below n has been read already
        for (int n = r; n < used; ++n) {
            const int f = fl[n];
            if (f & 4) {
                const int to = f >> 3;
                if ((f & 3) == MF_EXPANDED) {
                    const int32_t *ch = mc_child(T, g, n), *eN = mc_edge_n(T, g, n);
                    const float *eW = mc_edge_w(T, g, n), *eP = mc_edge_p(T, g, n);
                    int32_t *ch2 = mc_child(T, g, to), *eN2 = mc_edge_n(T, g, to);
                    float *eW2 = mc_edge_w(T, g, to), *eP2 = mc_edge_p(T, g, to);
                    for (int c = lane; c < T.Cp; c += width) {
                        const int j = ch[c];
                        const int fj = j >= 0 && j < used ? fl[j] : 0;
                        const int32_t x = eN[c];
                        const float w = eW[c], p = eP[c];
                        ch2[c] = (fj & 4) ? fj >> 3 : -1;
                        eN2[c] = x;
                        eW2[c] = w;
                        eP2[c] = p;
                    }
                }
                mc_sync();   // every lane has read the children's flags before lane 0 writes flags
                if (lead) {
                    nn[to] = nn[n];
                    fl[n] = f & 3;
                    fl[to] = f & 3;
                }
            }
            mc_sync();
        }
        if (lead) {
            nn[0] = en;
            m[MM_SIMS] = en;
            m[MM_VSUM] = (int32_t)(f_bits(ew) ^ 0x80000000u);
            m[MM_TOMOVE] = tn;
            uint32_t *rw = mc_rows(T, g);
#pragma unroll
            for (int y = 0; y < N; ++y) {
                rw[y] = black[y];
                rw[N + y] = empty[y];
            }
        }
    }
    mc_sync();   // every lane has read the meta
    if (lead) {
        m[MM_USED] = kept;
        m[MM_PENDING] = 0;
        m[MM_DEPTH] = 0;
        m[MM_NODE] = -1;
        m[MM_PARENT] = 0;
        m[MM_CELL] = 0;
    }
}

}  // namespace hexb
