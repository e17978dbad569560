// TEST INFRASTRUCTURE ONLY - host-side emulation of the tree-reuse kernel (hexb_mcts_advance_kernel).
//
// mcts_emu.cpp is included whole, so this library also carries every other emulated hexb_mcts_* call and the same emu_env struct
// from the same source: an EmuMCTS tree and an EmuBatch handle of tests/emu/emu.py can be passed here. The device code is the same
// per-root function the kernel runs (hex_gym_env_b200/csrc/hexb_mcts.cuh, mc_advance_root) with the one-lane host "warp".
#include "mcts_emu.cpp"

template <int N>
static void advance_n(const View &V, const MctsArgs &A) {
    Tree T;
    if (!mc_tree(A, N, V.G, T)) return;
    mc_write_first_playout(A);
    for (long long g = 0; g < V.G; ++g) mc_advance_root<N>(T, V, A, g);
}

extern "C" {

// hexb_mcts_advance on a host tree buffer
void emu_mcts_advance(void *h, uint8_t *tree, long long tree_bytes, long long first_playout, const uint8_t *root_mask) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    MctsArgs A;
    memset(&A, 0, sizeof(A));
    A.tree = tree;
    A.tree_bytes = (unsigned long long)tree_bytes;
    A.seed = e->base.seed;
    A.game_offset = (unsigned long long)e->base.game_offset;
    A.first_playout = first_playout;
    A.root_mask = root_mask;
    switch (e->N) {
#define X(n) \
    case n: advance_n<n>(V, A); break;
        HEXB_FOR_N(X)
#undef X
    }
}

}  // extern "C"
