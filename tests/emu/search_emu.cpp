// TEST INFRASTRUCTURE ONLY - host-side emulation of the tree-search kernels (hexb_copy_kernel, hexb_playout_kernel).
//
// Compiles the SAME per-game code the device runs (hex_gym_env_b200/csrc/hexb_search.cuh) with HEXB_HOST_EMU: a warp's ballot
// becomes a loop over its 32 lanes. The entry points take handles made by the step emulator (libhexb_emu.so, tests/emu/emu.py):
// hexb_emu.cpp is included whole, so emu_env here is the same struct from the same source. Lets the CPU suite check the copy
// conversion and the playouts against the oracle without a GPU.
#include "hexb_emu.cpp"

#include "../../hex_gym_env_b200/csrc/hexb_search.cuh"

template <int N>
static void playouts_n(const View &V, const PlayoutArgs &A) {
    for (long long g = 0; g < V.G; ++g) {
        uint32_t black[N], empty[N];
        const int to_move = (A.game_mask && !A.game_mask[g]) ? -1 : playout_rows<N>(V, g, black, empty);
        if (to_move < 0) {
            A.wins[g] = -1;
            continue;
        }
        int won = 0;
        for (int j = 0; j < A.num; ++j)
            won += playout_winner<N>(black, empty, to_move, A.seed, A.game_offset + (unsigned long long)g, (uint32_t)(A.first + j)) == to_move;
        A.wins[g] = won;
    }
}

extern "C" {

// hexb_copy_games: dst must be a raw emulator batch of the same N and variant
void emu_copy_games(void *dst_h, void *src_h, const int64_t *src_index, const int64_t *dst_index, long long count) {
    emu_env *dst = (emu_env *)dst_h, *src = (emu_env *)src_h;
    CopyArgs A;
    A.dst = dst->base.state;
    A.src = src->base.state;
    A.dst_G = dst->base.G;
    A.src_G = src->base.G;
    A.count = count;
    A.src_index = src_index;
    A.dst_index = dst_index;
    A.N = dst->N;
    const int C = A.N * A.N, W = (C + 31) / 32;
    for (long long i = 0; i < count; ++i) {   // one "warp" per pair
        long long s, d;
        if (!copy_pair(A, i, s, d)) continue;
        const uint32_t meta = copy_src_meta(A, s);
        const int tr = (meta & M_TRANSPOSED) ? 1 : 0;
        for (int w = 0; w < W; ++w) {
            uint32_t occ = 0;
            for (int lane = 0; lane < 32; ++lane) {
                const int c = 32 * w + lane;
                if (c < C && copy_cell(A, s, d, c, tr)) occ |= 1u << lane;
            }
            copy_store_rec(A, d, w, occ);
        }
        copy_store_rec(A, d, W, copy_meta(meta));
        copy_store_rec(A, d, W + 1, 0u);
    }
}

// hexb_playouts
void emu_playouts(void *h, int num_playouts, long long first_playout, const uint8_t *game_mask, int32_t *wins) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    PlayoutArgs A;
    A.seed = e->base.seed;
    A.game_offset = (unsigned long long)e->base.game_offset;
    A.first = first_playout;
    A.num = num_playouts;
    A.game_mask = game_mask;
    A.wins = wins;
    switch (e->N) {
#define X(n) \
    case n: playouts_n<n>(V, A); break;
        HEXB_FOR_N(X)
#undef X
    }
}

}  // extern "C"
