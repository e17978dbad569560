// hexb_search.cuh - tree-search primitives that are not on the step path: copying games into a bare HexGame (raw) batch
// (copy.deepcopy(env.simulator)) and Monte-Carlo playouts from the current position. Written per element / per game like
// hexb_views.cuh, so that the kernels are thin wrappers and the host emulator (tests/emu) runs the same code.
#pragma once
#include "hexb_views.cuh"

namespace hexb {

// ---------------------------------------------------------------------------------------------- copy_games
// Pair i copies src game src_index[i] into dst game dst_index[i] (null index = identity). dst is a raw handle with the same N
// and variant. An env game whose agent is WHITE (M_TRANSPOSED) is stored transposed with R = WHITE: the copy is converted to
// true coordinates and colours, which is how a raw game stores itself (HexGame.__init__ state, HexGame.py:21-68,
// HexSingleGame.py:26-71).
struct CopyArgs {
    uint8_t *dst;
    const uint8_t *src;
    long long dst_G, src_G, count;
    const int64_t *src_index, *dst_index;
    int N;
};

// false: an index is out of range and the pair writes nothing
HEXB_HD bool copy_pair(const CopyArgs &A, long long i, long long &s, long long &d) {
    s = A.src_index ? (long long)A.src_index[i] : i;
    d = A.dst_index ? (long long)A.dst_index[i] : i;
    return s >= 0 && s < A.src_G && d >= 0 && d < A.dst_G;
}

HEXB_HD uint32_t copy_src_meta(const CopyArgs &A, long long s) {
    const int C = A.N * A.N, W = (C + 31) / 32;
    return reinterpret_cast<const uint32_t *>(A.src + rec_offset(s, C))[W * kRecStride];
}

// Label byte of dst cell c (true row-major); returns whether it holds a stone (the occupancy bit). tr: the src game is stored
// transposed, so its stored cell (x, y) is true cell (y, x) and its owner bit is the other colour.
HEXB_HD bool copy_cell(const CopyArgs &A, long long s, long long d, int c, int tr) {
    const int N = A.N, C = N * N;
    const int y = c / N, x = c - y * N;
    uint32_t b = A.src[labels_offset(s, C) + (tr ? x * N + y : c)];
    if (tr && b) b ^= 0x80u;
    A.dst[labels_offset(d, C) + c] = (uint8_t)b;
    return b != 0u;
}

// The raw game's meta word: the stored sides swapped back for a transposed game (counters, far-edge flags, winner code, side to
// move), the env-only bits dropped (agent orientation, agent-ended, illegal-move end) - what a raw handle's own import produces
// for the same position, with the exact counters.
HEXB_HD uint32_t copy_meta(uint32_t m) {
    if (m & M_TRANSPOSED) {
        const uint32_t cr = (m >> M_CTR_R_SHIFT) & 0xffu, cc = (m >> M_CTR_C_SHIFT) & 0xffu;
        const uint32_t w = (m & M_WIN_MASK) >> M_WIN_SHIFT;
        uint32_t o = m & ~(0xffffu | M_FAR_R1 | M_FAR_C1 | M_WIN_MASK);
        o |= (cc << M_CTR_R_SHIFT) | (cr << M_CTR_C_SHIFT);
        if (m & M_FAR_R1) o |= M_FAR_C1;
        if (m & M_FAR_C1) o |= M_FAR_R1;
        o |= (w == 0u ? 0u : 3u - w) << M_WIN_SHIFT;
        m = o ^ M_TOMOVE;
    }
    return m & ~(M_TRANSPOSED | M_AGENT_ENDED | M_INVALID);
}

HEXB_HD void copy_store_rec(const CopyArgs &A, long long d, int w, uint32_t v) {
    reinterpret_cast<uint32_t *>(A.dst + rec_offset(d, A.N * A.N))[w * kRecStride] = v;
}

// ---------------------------------------------------------------------------------------------- playouts
struct PlayoutArgs {
    unsigned long long seed, game_offset;
    long long first;          // first playout index p
    int num;                  // playouts per game
    const uint8_t *game_mask; // [G] nullable
    int32_t *wins;            // [G] playouts won by the side to move, -1 = no playouts
};

// Playout p of global game g: from the current position with the side to move first, colours alternating, ply k plays the
// int(u * n_empty)-th empty cell in true row-major order (random_policy, minihex/__init__.py:8-12) with u built like draw01 from
// Philox4x32-10 at counter (k, g_lo, g_hi, p + 1): c3 = 0 is the env streams', so playout streams never meet them. Stones are
// never removed and a full Hex board has exactly one winner, so the board is filled to the end and its connectivity tested once.
HEXB_HD double playout_draw(unsigned long long seed, unsigned long long game, uint32_t k, uint32_t p) {
    uint32_t a, b;
    philox4x32_10(k, (uint32_t)game, (uint32_t)(game >> 32), p + 1u, (uint32_t)seed, (uint32_t)(seed >> 32), a, b);
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// True-orientation rows of game g: black[y] / empty[y] bit x = cell (y, x). Returns the true colour to move, or -1 when the game
// has no playouts (never reset, or finished).
template <int N>
HEXB_HD int playout_rows(const View &V, long long g, uint32_t (&black)[N], uint32_t (&empty)[N]) {
    const uint32_t meta = view_meta(V, g);
    if (!(meta & M_LIVE) || (meta & M_DONE)) return -1;
    const int tr = (meta & M_TRANSPOSED) ? 1 : 0;
    const uint8_t *L = view_labels(V, g);
#pragma unroll
    for (int y = 0; y < N; ++y) {
        uint32_t bl = 0, em = 0;
#pragma unroll
        for (int x = 0; x < N; ++x) {
            const uint32_t b = L[tr ? x * N + y : y * N + x];
            em |= (b == 0u ? 1u : 0u) << x;
            bl |= (b != 0u && (int)(b >> 7) == tr ? 1u : 0u) << x;   // stored owner R is true BLACK unless transposed
        }
        black[y] = bl;
        empty[y] = em;
    }
    return ((meta & M_TOMOVE) ? 1 : 0) ^ tr;
}

HEXB_HD uint32_t brev32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __brev(v);
#else
    v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
    v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
    v = ((v >> 4) & 0x0f0f0f0fu) | ((v & 0x0f0f0f0fu) << 4);
    v = ((v >> 8) & 0x00ff00ffu) | ((v & 0x00ff00ffu) << 8);
    return (v >> 16) | (v << 16);
#endif
}

// the runs of m (one board row) that contain a seed bit (s within m): adding s to m carries through each run from its lowest seed
// upwards; the bit-reversed sum does the same downwards
HEXB_HD uint32_t row_fill(uint32_t m, uint32_t s) {
    const uint32_t up = (((m + s) ^ m) & m) | s;
    const uint32_t rm = brev32(m), rs = brev32(s);
    const uint32_t dn = brev32((((rm + rs) ^ rm) & rm) | rs);
    return up | dn;
}

// BLACK connects row 0 to row N-1 on a full board (else WHITE connects the columns). Neighbours of (y, x): the 3x3 window minus
// (-1,-1) and (+1,+1) (HexGame.py:124-142): (y+1, x-1), (y+1, x) below, (y-1, x), (y-1, x+1) above.
template <int N>
HEXB_HD bool black_connects(const uint32_t (&black)[N]) {
    uint32_t r[N];
    r[0] = black[0];
#pragma unroll
    for (int y = 1; y < N; ++y) r[y] = 0u;
    bool changed = true;
    while (changed) {
        changed = false;
#pragma unroll
        for (int y = 1; y < N; ++y) {
            const uint32_t nr = row_fill(black[y], ((r[y - 1] | (r[y - 1] >> 1)) & black[y]) | r[y]);
            changed |= nr != r[y];
            r[y] = nr;
        }
        if (r[N - 1]) return true;
#pragma unroll
        for (int y = N - 2; y >= 0; --y) {
            const uint32_t nr = row_fill(black[y], ((r[y + 1] | (r[y + 1] << 1)) & black[y]) | r[y]);
            changed |= nr != r[y];
            r[y] = nr;
        }
    }
    return false;
}

// k-th (0-based) set bit of z (k < popcount(z))
HEXB_HD int nth_set_bit(uint32_t z, int k) {
    int pos = 0, c;
    c = popc32(z & 0xffffu); if (k >= c) { k -= c; pos += 16; z >>= 16; }
    c = popc32(z & 0xffu);   if (k >= c) { k -= c; pos += 8;  z >>= 8; }
    c = popc32(z & 0xfu);    if (k >= c) { k -= c; pos += 4;  z >>= 4; }
    c = popc32(z & 0x3u);    if (k >= c) { k -= c; pos += 2;  z >>= 2; }
    c = (int)(z & 1u);       if (k >= c) { pos += 1; }
    return pos;
}

// One playout from rows (black0, empty0) with true colour `to_move` first; returns the winning true colour (0 BLACK, 1 WHITE).
// Rows are selected by unrolled compare-and-mask, never by a run-time index, so that the arrays stay in registers.
template <int N>
HEXB_HD int playout_winner(const uint32_t (&black0)[N], const uint32_t (&empty0)[N], int to_move, unsigned long long seed,
                           unsigned long long game, uint32_t p) {
    uint32_t black[N], empty[N];
    int n = 0;
#pragma unroll
    for (int y = 0; y < N; ++y) {
        black[y] = black0[y];
        empty[y] = empty0[y];
        n += popc32(empty0[y]);
    }
    for (uint32_t k = 0; n > 0; ++k, --n) {
        int left = choice_of(playout_draw(seed, game, k, p), n);
        uint32_t z = 0u;
        int row = -1, kk = 0;
#pragma unroll
        for (int y = 0; y < N; ++y) {
            const int c = popc32(empty[y]);
            if (row < 0 && left < c) { row = y; z = empty[y]; kk = left; }
            left -= c;
        }
        const uint32_t bit = 1u << nth_set_bit(z, kk);
        const uint32_t bl = ((k & 1u) ? 1 - to_move : to_move) == 0 ? bit : 0u;
#pragma unroll
        for (int y = 0; y < N; ++y) {
            const uint32_t m = y == row ? bit : 0u;
            empty[y] &= ~m;
            black[y] |= m & bl;
        }
    }
    return black_connects<N>(black) ? 0 : 1;
}

}  // namespace hexb
