// hexb_step_inst.cu - everything of libhexb.so that is templated on the board size, for ONE size (the step kernels of
// hexb_step.cuh in their one-warp and 4-warp-per-chunk forms, and the kernels below): compiled once per
// N = 3..19 with -DHEXB_INST_N=n (hex_gym_env_b200/_native.py builds the 17 objects in parallel and links them with
// hexb_kernels.cu). nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo.
#ifndef HEXB_INST_N
#error "compile with -DHEXB_INST_N=<board size>"
#endif
#include "hexb_step.cuh"

#define HEXB_CAT_(a, b) a##b
#define HEXB_CAT(a, b) HEXB_CAT_(a, b)

template <int N>
__global__ void hexb_sample_kernel(View V, int view, const double *u, int32_t *out) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < V.G) sample_at<N>(V, view, g, u, out);
}
template <int N>
__global__ void hexb_import_kernel(Params P, const int8_t *board_true, const int8_t *to_move, const uint8_t *import_mask) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < P.G) import_game<N>(P, g, board_true, to_move, import_mask);
}

// hexb_playouts_policy: one warp per game, lane l takes playouts first + l, first + l + 32, ... (every playout of a game fills the
// same number of cells, so the lanes stay converged until the connectivity test)
template <int N, int POLICY>
__global__ void __launch_bounds__(256) hexb_playout_kernel(View V, PlayoutArgs A) {
    const int lane = threadIdx.x & 31;
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= V.G) return;
    uint32_t black[N], empty[N];
    const int to_move = (A.game_mask && !A.game_mask[g]) ? -1 : playout_rows<N>(V, g, black, empty);
    if (to_move < 0) {
        if (lane == 0) A.wins[g] = -1;
        return;
    }
    const unsigned long long gid = A.game_offset + (unsigned long long)g;
    int won = 0;
    for (int j = lane; j < A.num; j += 32)
        won += playout_winner<N, POLICY>(black, empty, to_move, A.seed, gid, (uint32_t)(A.first + j), -1) == to_move;
    won = __reduce_add_sync(0xffffffffu, won);
    if (lane == 0) A.wins[g] = won;
}

// hexb_mcts_*: the tree search of hexb_mcts.cuh. init: one thread per root (thread 0 also writes the header); the others: one warp
// per root, all S simulations of the fused search in one launch, and advance's subtree compaction.
template <int N>
__global__ void __launch_bounds__(128) hexb_mcts_init_kernel(View V, MctsArgs A) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) mc_write_header(A, N, V.G);
    if (g < V.G) mc_init_root<N>(V, A, g);
}
// 168 registers: the path rows, the playout's own copy and the selection state without a spill at N = 19 (ptxas -v), for both
// playout policies
template <int N, int POLICY>
__global__ void __maxnreg__(168) hexb_mcts_search_kernel(View V, MctsArgs A) {
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    Tree T;
    if (g < V.G && mc_tree(A, N, V.G, T)) mc_search_root<N, POLICY>(T, A, V.variant, g);
}
template <int N>
__global__ void __launch_bounds__(128) hexb_mcts_select_kernel(View V, MctsArgs A) {
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    Tree T;
    if (g < V.G && mc_tree(A, N, V.G, T)) mc_select_root<N>(T, V, A, g);
}
template <int N>
__global__ void __launch_bounds__(128) hexb_mcts_expand_kernel(View V, MctsArgs A) {
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    Tree T;
    if (g < V.G && mc_tree(A, N, V.G, T)) mc_expand_root<N>(T, V, A, g);
}
template <int N>
__global__ void __launch_bounds__(128) hexb_mcts_root_kernel(View V, MctsArgs A) {
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    Tree T;
    if (g < V.G && mc_tree(A, N, V.G, T)) mc_root_out(T, V.variant, A, g);
}
// advance: thread 0 writes the header's first_playout once the header has been checked; one warp per root
template <int N>
__global__ void __launch_bounds__(128) hexb_mcts_advance_kernel(View V, MctsArgs A) {
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    Tree T;
    if (g < V.G && mc_tree(A, N, V.G, T)) {
        if (blockIdx.x == 0 && threadIdx.x == 0) mc_write_first_playout(A);
        mc_advance_root<N>(T, V, A, g);
    }
}

int HEXB_CAT(hexb_launch_tile_, HEXB_INST_N)(const hexb_env *e, const Params &P, cudaStream_t s) { return launch_tile<HEXB_INST_N>(e, P, s); }

int HEXB_CAT(hexb_launch_sample_, HEXB_INST_N)(const View &V, int view, const double *u, int32_t *out, cudaStream_t s) {
    hexb_sample_kernel<HEXB_INST_N><<<(unsigned)((V.G + 127) / 128), 128, 0, s>>>(V, view, u, out);
    CK(cudaGetLastError());
    return HEXB_OK;
}

int HEXB_CAT(hexb_launch_import_, HEXB_INST_N)(const Params &P, const int8_t *board_true, const int8_t *to_move, const uint8_t *import_mask,
                                               cudaStream_t s) {
    hexb_import_kernel<HEXB_INST_N><<<(unsigned)((P.G + 127) / 128), 128, 0, s>>>(P, board_true, to_move, import_mask);
    CK(cudaGetLastError());
    return HEXB_OK;
}

// policy: PLAYOUT_RANDOM or PLAYOUT_BRIDGE (checked by the caller)
int HEXB_CAT(hexb_launch_playouts_, HEXB_INST_N)(const View &V, const PlayoutArgs &A, int policy, cudaStream_t s) {
    const unsigned blocks = (unsigned)((V.G + 7) / 8);
    if (policy == PLAYOUT_BRIDGE) hexb_playout_kernel<HEXB_INST_N, PLAYOUT_BRIDGE><<<blocks, 256, 0, s>>>(V, A);
    else hexb_playout_kernel<HEXB_INST_N, PLAYOUT_RANDOM><<<blocks, 256, 0, s>>>(V, A);
    CK(cudaGetLastError());
    return HEXB_OK;
}

// policy: the fused search's playout policy (MCTS_SEARCH only)
int HEXB_CAT(hexb_launch_mcts_, HEXB_INST_N)(int op, const View &V, const MctsArgs &A, int policy, cudaStream_t s) {
    const unsigned warps = (unsigned)((V.G + 3) / 4), threads = (unsigned)((V.G + 127) / 128);
    switch (op) {
        case MCTS_INIT: hexb_mcts_init_kernel<HEXB_INST_N><<<threads, 128, 0, s>>>(V, A); break;
        case MCTS_SEARCH:
            if (policy == PLAYOUT_BRIDGE) hexb_mcts_search_kernel<HEXB_INST_N, PLAYOUT_BRIDGE><<<warps, 128, 0, s>>>(V, A);
            else hexb_mcts_search_kernel<HEXB_INST_N, PLAYOUT_RANDOM><<<warps, 128, 0, s>>>(V, A);
            break;
        case MCTS_SELECT: hexb_mcts_select_kernel<HEXB_INST_N><<<warps, 128, 0, s>>>(V, A); break;
        case MCTS_EXPAND: hexb_mcts_expand_kernel<HEXB_INST_N><<<warps, 128, 0, s>>>(V, A); break;
        case MCTS_ROOT: hexb_mcts_root_kernel<HEXB_INST_N><<<warps, 128, 0, s>>>(V, A); break;
        case MCTS_ADVANCE: hexb_mcts_advance_kernel<HEXB_INST_N><<<warps, 128, 0, s>>>(V, A); break;
        default: return HEXB_ERR_ARG;
    }
    CK(cudaGetLastError());
    return HEXB_OK;
}
