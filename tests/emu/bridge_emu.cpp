// TEST INFRASTRUCTURE ONLY - host-side emulation of the playout kernels of both policies (hexb_playout_kernel<N, policy>,
// hexb_mcts_search_kernel<N, policy>: hexb_playouts_policy, hexb_mcts_search_policy).
//
// mcts_emu.cpp is included whole, so this library also carries every other emulated hexb_mcts_* call and the same emu_env struct
// from the same source: an EmuMCTS tree and an EmuBatch handle of tests/emu/emu.py can be passed here. The device code is the same
// per-game and per-root code the kernels run (hex_gym_env_b200/csrc/hexb_search.cuh, hexb_mcts.cuh) with the one-lane host "warp".
#include "mcts_emu.cpp"

template <int N, int POLICY>
static void playouts_policy_n(const View &V, const PlayoutArgs &A) {
    for (long long g = 0; g < V.G; ++g) {
        uint32_t black[N], empty[N];
        const int to_move = (A.game_mask && !A.game_mask[g]) ? -1 : playout_rows<N>(V, g, black, empty);
        if (to_move < 0) {
            A.wins[g] = -1;
            continue;
        }
        int won = 0;
        for (int j = 0; j < A.num; ++j)
            won += playout_winner<N, POLICY>(black, empty, to_move, A.seed, A.game_offset + (unsigned long long)g, (uint32_t)(A.first + j),
                                             -1) == to_move;
        A.wins[g] = won;
    }
}

template <int N, int POLICY>
static void search_policy_n(const View &V, const MctsArgs &A) {
    Tree T;
    if (!mc_tree(A, N, V.G, T)) return;
    for (long long g = 0; g < V.G; ++g) mc_search_root<N, POLICY>(T, A, V.variant, g);
}

extern "C" {

// hexb_playouts_policy (policy PLAYOUT_RANDOM or PLAYOUT_BRIDGE)
void emu_playouts_policy(void *h, int num_playouts, long long first_playout, int policy, const uint8_t *game_mask, int32_t *wins) {
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
    case n: policy == PLAYOUT_BRIDGE ? playouts_policy_n<n, PLAYOUT_BRIDGE>(V, A) : playouts_policy_n<n, PLAYOUT_RANDOM>(V, A); break;
        HEXB_FOR_N(X)
#undef X
    }
}

// hexb_mcts_search_policy on a host tree buffer
void emu_mcts_search_policy(void *h, uint8_t *tree, long long tree_bytes, int sims, int playouts, int policy) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    MctsArgs A;
    memset(&A, 0, sizeof(A));
    A.tree = tree;
    A.tree_bytes = (unsigned long long)tree_bytes;
    A.seed = e->base.seed;
    A.game_offset = (unsigned long long)e->base.game_offset;
    A.sims = sims;
    A.playouts = playouts;
    switch (e->N) {
#define X(n) \
    case n: policy == PLAYOUT_BRIDGE ? search_policy_n<n, PLAYOUT_BRIDGE>(V, A) : search_policy_n<n, PLAYOUT_RANDOM>(V, A); break;
        HEXB_FOR_N(X)
#undef X
    }
}

}  // extern "C"
