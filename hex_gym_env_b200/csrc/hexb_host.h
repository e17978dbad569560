// hexb_host.h - host-side declarations shared by the translation units of libhexb.so (not part of the C ABI).
//
// The library is built from one object per board size (hexb_step_inst.cu compiled with -DHEXB_INST_N=n: every instantiation of
// the step kernels for that N (one warp or a CTA of 4 warps per chunk) plus the small per-N kernels: sampler, import, playouts, tree search) and hexb_kernels.cu (the C ABI, the size-independent kernels and
// the dispatch tables). The per-N objects are independent, so hex_gym_env_b200/_native.py compiles them in parallel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../include/hexb.h"
#include "hexb_mcts.cuh"

#define HEXB_LOCAL __attribute__((visibility("hidden")))

#define HEXB_HOST_SLICES 6   // pieces the packed words of a host-buffer step travel in (host threads expand piece k while k+1 is in flight)

struct hexb_env {
    hexb_config cfg;
    hexb::Params base;   // state pointers + config, I/O pointers null
    int launch_form;     // hexb_set_launch_form: 0 = chosen by launch depth, 1 / 4 = warps per 32-game chunk
    // ---- host-buffer step (hexb_step_host*): events, staging and the adaptive DMA / packed split
    cudaEvent_t host_ev, host_ev_dma0, host_ev_slice[HEXB_HOST_SLICES];   // all copies done; start of the DMA part; each packed slice arrived
    int host_pending, host_adapt, host_frac_fixed;
    double host_dma_frac;          // share of the games whose obs / mask rows travel as plain bytes by DMA
    double host_dma_bytes;
    double host_t0_ms;                                   // start of the running synchronous call
    int host_tune_calls;                                 // position in the split search (tune_next in hexb_kernels.cu)
    double host_tune_ms[7][3], host_tune_best, host_tune_best_ms;
    long long host_plan_words, host_plan_first, host_slice_lo[HEXB_HOST_SLICES], host_slice_hi[HEXB_HOST_SLICES];
    uint32_t *host_packed;         // pinned staging of the packed words (cudaHostAlloc, owned by the handle)
    const uint32_t *host_packed_src;
    int8_t *host_obs;
    uint8_t *host_mask;
};

HEXB_LOCAL int hexb_cuda_fail(cudaError_t e);   // records the code for hexb_last_cuda_error, returns HEXB_ERR_CUDA
#define CK(call)                                       \
    do {                                               \
        cudaError_t e_ = (call);                       \
        if (e_ != cudaSuccess) return hexb_cuda_fail(e_); \
    } while (0)

enum : int { MCTS_INIT = 0, MCTS_SEARCH, MCTS_SELECT, MCTS_EXPAND, MCTS_ROOT, MCTS_ADVANCE };   // op of hexb_launch_mcts_<n>

// per-board-size entry points, defined by hexb_step_inst.cu
#define HEXB_FOR_N(X) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19)
#define HEXB_DECL_N(n)                                                                                                      \
    HEXB_LOCAL int hexb_launch_tile_##n(const hexb_env *e, const hexb::Params &P, cudaStream_t s);                          \
    HEXB_LOCAL int hexb_launch_sample_##n(const hexb::View &V, int view, const double *u, int32_t *out, cudaStream_t s);     \
    HEXB_LOCAL int hexb_launch_import_##n(const hexb::Params &P, const int8_t *board_true, const int8_t *to_move,           \
                                          const uint8_t *import_mask, cudaStream_t s);                                      \
    HEXB_LOCAL int hexb_launch_playouts_##n(const hexb::View &V, const hexb::PlayoutArgs &A, cudaStream_t s);             \
    HEXB_LOCAL int hexb_launch_mcts_##n(int op, const hexb::View &V, const hexb::MctsArgs &A, cudaStream_t s);
HEXB_FOR_N(HEXB_DECL_N)
#undef HEXB_DECL_N
