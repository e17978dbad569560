// TEST INFRASTRUCTURE ONLY - host-side emulation of the tree-search kernels (hexb_mcts_*_kernel).
//
// Compiles the SAME per-root code the device runs (hex_gym_env_b200/csrc/hexb_mcts.cuh) with HEXB_HOST_EMU: the search's warp
// becomes one lane that owns every cell and every path entry, so its shuffles become loops. The entry points take handles made by
// the step emulator (libhexb_emu.so, tests/emu/emu.py): hexb_emu.cpp is included whole, so emu_env here is the same struct from the
// same source. Lets the CPU suite check the whole tree against the oracle (oracle/mcts.py) without a GPU.
#include "hexb_emu.cpp"

#include "../../hex_gym_env_b200/csrc/hexb_mcts.cuh"

// the tree buffer is host memory; op as hexb_launch_mcts_<n>
enum { OP_INIT = 0, OP_SEARCH, OP_SELECT, OP_EXPAND, OP_ROOT };

template <int N>
static void mcts_n(int op, const View &V, const MctsArgs &A) {
    if (op == OP_INIT) {
        mc_write_header(A, N, V.G);
        for (long long g = 0; g < V.G; ++g) mc_init_root<N>(V, A, g);
        return;
    }
    Tree T;
    if (!mc_tree(A, N, V.G, T)) return;
    for (long long g = 0; g < V.G; ++g) {
        if (op == OP_SEARCH) mc_search_root<N>(T, A, V.variant, g);
        else if (op == OP_SELECT) mc_select_root<N>(T, V, A, g);
        else if (op == OP_EXPAND) mc_expand_root<N>(T, V, A, g);
        else mc_root_out(T, V.variant, A, g);
    }
}

extern "C" {

long long emu_mcts_tree_bytes(int N, long long G, int max_nodes) { return 128 + mc_root_bytes(N, max_nodes) * G; }

// every argument of every hexb_mcts_* call; the ones op does not use are ignored
void emu_mcts(void *h, int op, uint8_t *tree, long long tree_bytes, int max_nodes, double c_puct, double fpu, long long first_playout,
              const uint8_t *root_mask, int sims, int playouts, void *leaf_obs, uint8_t *leaf_mask, uint8_t *pending,
              const float *priors, const float *values, int32_t *visits, float *q, float *value, int32_t *nodes_used) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    MctsArgs A;
    memset(&A, 0, sizeof(A));
    A.tree = tree;
    A.tree_bytes = (unsigned long long)tree_bytes;
    A.seed = e->base.seed;
    A.game_offset = (unsigned long long)e->base.game_offset;
    A.max_nodes = max_nodes;
    A.c_puct = (float)c_puct;
    A.fpu = (float)fpu;
    A.first_playout = first_playout;
    A.root_mask = root_mask;
    A.sims = sims;
    A.playouts = playouts;
    A.leaf_obs = leaf_obs;
    A.leaf_mask = leaf_mask;
    A.pending = pending;
    A.priors = priors;
    A.values = values;
    A.visits = visits;
    A.q = q;
    A.value = value;
    A.nodes_used = nodes_used;
    switch (e->N) {
#define X(n) \
    case n: mcts_n<n>(op, V, A); break;
        HEXB_FOR_N(X)
#undef X
    }
}

}  // extern "C"
