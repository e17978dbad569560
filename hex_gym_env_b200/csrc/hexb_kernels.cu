// hexb_kernels.cu - the C ABI (include/hexb.h) of the batched Hex simulator and its size-independent sm_100a kernels.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo (hex_gym_env_b200/_native.py: this file, one object per board
// size from hexb_step_inst.cu, and the host-only hexb_hostpack.cpp, linked into libhexb.so).
//
// Kernel inventory (SURVEY.md section 2.3):
//   K1/K2/K3  hexb_step_kernel<N> / hexb_coop_kernel<N>  (hexb_step.cuh) MODE_RESET / MODE_STEP / MODE_PLY / MODE_HALF, T steps
//             per launch for hexb_rollout; one warp per 32-game chunk, or a CTA of 4 warps per chunk for sub-wave launches
//   K4        hexb_sample_kernel<N>   standalone k-th-empty-cell sampler (hexb_step_inst.cu)
//   K5        hexb_encode_kernel      standalone observation + mask encoder (either view)
//   K6        hexb_export_kernel / hexb_import_kernel<N>   reference-layout dump / preset boards
//   K7        statistics: warp __reduce_add_sync + one atomic per chunk and counter (striped); hexb_stats sums the stripes
//   K8        hexb_masked_sample_kernel   masked categorical sampling (the rollout feed)
//   K9        hexb_gae_kernel         GAE(lambda) advantages / returns over a [T,G] rollout (SB3 RolloutBuffer semantics)
//   K10       hexb_pack_obs_kernel    2-bit observation transport for hexb_step_host_packed
//   K11       hexb_copy_kernel        copy.deepcopy(env.simulator) into a raw batch, one warp per copied game (hexb_search.cuh)
//   K12       hexb_playout_kernel<N>  random playouts from the current position, one warp per game (hexb_step_inst.cu)
//   K13       hexb_mcts_*_kernel<N>   batched PUCT tree search: init, fused search, select, expand, root readout, advance (hexb_mcts.cuh)
#include <cuda.h>   // types of the driver's virtual-memory API only (entry points come from cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <map>
#include <mutex>

#include "hexb_host.h"

using namespace hexb;

// ------------------------------------------------------------------------------------------------ small kernels (hexb_views.cuh)
__global__ void hexb_encode_kernel(View V, int view, int8_t *obs, uint8_t *mask) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V.G * V.N * V.N) encode_at(V, view, i, obs, mask);
}
__global__ void hexb_export_kernel(View V, double *board, double *regions, double *counter, int8_t *cur, uint8_t *done,
                                   int8_t *winner, int8_t *agent, uint32_t *draws) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V.G * 2 * (V.N + 2) * (V.N + 2)) export_at(V, i, board, regions, counter, cur, done, winner, agent, draws);
}

__global__ void hexb_import_labels_kernel(Params P, int N, const int8_t *board_true, const uint8_t *planes, const int8_t *to_move,
                                          const uint8_t *import_mask) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < P.G) import_labels_game(P, N, g, board_true, planes, to_move, import_mask);
}

// K11: one warp per copied game; lane l writes cells l, l + 32, ... and the ballot of their stones is the occupancy word
__global__ void __launch_bounds__(128) hexb_copy_kernel(CopyArgs A) {
    const int lane = threadIdx.x & 31;
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    long long s, d;
    if (i >= A.count || !copy_pair(A, i, s, d)) return;
    const int C = A.N * A.N, W = (C + 31) / 32;
    const uint32_t meta = copy_src_meta(A, s);
    const int tr = (meta & M_TRANSPOSED) ? 1 : 0;
    for (int w = 0; w < W; ++w) {
        const int c = 32 * w + lane;
        const uint32_t occ = __ballot_sync(0xffffffffu, c < C && copy_cell(A, s, d, c, tr));
        if (lane == 0) copy_store_rec(A, d, w, occ);
    }
    if (lane == 0) {
        copy_store_rec(A, d, W, copy_meta(meta));
        copy_store_rec(A, d, W + 1, 0u);   // draws: a raw game has no stream
    }
}

__global__ void hexb_stats_kernel(const long long *src, int64_t *dst) {
    if (threadIdx.x < 8) {
        long long v = 0;
        for (int s = 0; s < kStatStripes; ++s) v += src[8 * s + threadIdx.x];
        dst[threadIdx.x] = (int64_t)v;
    }
}

// K8: masked categorical sampling, one warp per game. Cells are dealt to lanes in blocks of 32 (cell = 32*k + lane), so a
// block's inclusive scan over lanes continues the running CDF in cell order.
__global__ void __launch_bounds__(128) hexb_masked_sample_kernel(const float *__restrict__ logits, const uint8_t *__restrict__ mask,
                                                                 const double *__restrict__ u, long long G, int C, int32_t *actions,
                                                                 float *logp, float *entropy) {
    constexpr uint32_t FULL = 0xffffffffu;
    constexpr int KMAX = (HEXB_MAX_BOARD * HEXB_MAX_BOARD + 31) / 32;
    const int lane = threadIdx.x & 31;
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= G) return;
    const float *lg = logits + g * C;
    const uint8_t *mk = mask + g * C;
    const int K = (C + 31) >> 5;
    float l[KMAX];
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
        const int c = 32 * k + lane;
        l[k] = (k < K && c < C && mk[c]) ? lg[c] : -INFINITY;
        mx = fmaxf(mx, l[k]);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, o));
    if (mx == -INFINITY) {  // no legal cell
        if (lane == 0) {
            if (actions) actions[g] = -1;
            if (logp) logp[g] = 0.f;
            if (entropy) entropy[g] = 0.f;
        }
        return;
    }
    float e[KMAX], z = 0.f, sel = 0.f;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
        e[k] = (l[k] == -INFINITY) ? 0.f : __expf(l[k] - mx);
        z += e[k];
        sel += e[k] * ((l[k] == -INFINITY) ? 0.f : (l[k] - mx));
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        z += __shfl_xor_sync(FULL, z, o);
        sel += __shfl_xor_sync(FULL, sel, o);
    }
    const float logz = __logf(z);
    const float target = (float)(u[g] * (double)z);
    float run = 0.f;
    int pick = -1, last_legal = -1;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
        if (k < K) {
            float s = e[k];  // inclusive scan over lanes
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float t = __shfl_up_sync(FULL, s, o);
                if (lane >= o) s += t;
            }
            const float cum = run + s;
            const uint32_t hit = __ballot_sync(FULL, e[k] > 0.f && cum > target);
            const uint32_t legal = __ballot_sync(FULL, e[k] > 0.f);
            if (pick < 0 && hit) pick = 32 * k + (__ffs(hit) - 1);
            if (legal) last_legal = 32 * k + (31 - __clz(legal));
            run += __shfl_sync(FULL, s, 31);
        }
    }
    if (pick < 0) pick = last_legal;  // u*z rounded up to the total: the last legal cell
    const int pk = pick >> 5, pl = pick & 31;
    float lp = 0.f;
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
        if (k == pk) lp = l[k];
    lp = __shfl_sync(FULL, lp, pl) - mx - logz;
    if (lane == 0) {
        if (actions) actions[g] = pick;
        if (logp) logp[g] = lp;
        if (entropy) entropy[g] = logz - sel / z;
    }
}


// K9: generalised advantage estimation, one thread per game, backward over the T steps of a rollout. Exactly the recurrence of
// stable-baselines3's RolloutBuffer.compute_returns_and_advantage (2.2.1; what MaskablePPO runs after collect_rollouts in the
// reference's training scripts, scripts/experiments/*.py:40-47): a finished episode (done[t]) cuts the bootstrap and the trace.
// Single-precision, operation for operation like the eager PyTorch loop it replaces (no fused multiply-add), so that both agree
// to the last bit on the same inputs. Reads and writes are coalesced over games.
__global__ void hexb_gae_kernel(const float *__restrict__ rewards, const float *__restrict__ values, const uint8_t *__restrict__ dones,
                                int T, long long G, float gamma, float gl, float *__restrict__ adv, float *__restrict__ ret) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    float last = 0.f;
    float v_next = values[(long long)T * G + g];
    for (int t = T - 1; t >= 0; --t) {
        const long long i = (long long)t * G + g;
        const float nt = dones[i] ? 0.f : 1.f;
        const float v = values[i];
        // delta = r + gamma * V(t+1) * nonterminal - V(t);  last = delta + gamma * lambda * nonterminal * last
        const float delta = __fsub_rn(__fadd_rn(rewards[i], __fmul_rn(__fmul_rn(gamma, v_next), nt)), v);
        last = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nt), last));
        adv[i] = last;
        if (ret) ret[i] = __fadd_rn(last, v);
        v_next = v;
    }
}

// K10: observation bytes -> 2 bits per cell (code = byte & 3: variant B -1/0/+1 -> 3/0/1, variant A 0/1/2), 16 cells per thread
// and output word, flat over the [G*C] cells. The host side of hexb_step_host_packed expands them again (hexb_hostpack.cpp).
__global__ void hexb_pack_obs_kernel(const uint4 *__restrict__ obs16, long long n_words, uint32_t *__restrict__ packed) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    const uint4 x = obs16[i];
    const uint32_t w[4] = {x.x, x.y, x.z, x.w};
    uint32_t out = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t v = w[k] & 0x03030303u;   // one 2-bit code per byte
        const uint32_t b = (v | (v >> 6) | (v >> 12) | (v >> 18)) & 0xffu;   // the four codes side by side
        out |= b << (8 * k);
    }
    packed[i] = out;
}
// ------------------------------------------------------------------------------------------------ host side
static thread_local int g_last_cuda = 0;
int hexb_cuda_fail(cudaError_t e) {
    g_last_cuda = (int)e;
    return HEXB_ERR_CUDA;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static bool cfg_ok(const hexb_config *c) {
    if (!c) return false;
    if (c->board_size < HEXB_MIN_BOARD || c->board_size > HEXB_MAX_BOARD) return false;
    if (c->variant != HEXB_VARIANT_A && c->variant != HEXB_VARIANT_B) return false;
    if (c->num_games < 1 || c->game_offset < 0) return false;
    if (c->agent_mode < 0 || c->agent_mode > 2) return false;
    if (c->variant == HEXB_VARIANT_A && c->agent_mode != HEXB_AGENT_BLACK) return false;
    if (c->pool_size < 0 || (c->manual_opponent && c->raw)) return false;
    if (c->obs_dtype != HEXB_OBS_I8 && c->obs_dtype != HEXB_OBS_F32) return false;
    return true;
}

struct Layout {
    long long Gpad;
    size_t stats_off, total;   // the chunks (labels + records of 32 games each) start at offset 0; the statistics follow
};
static Layout layout_of(const hexb_config *c) {
    Layout L;
    const long long C = (long long)c->board_size * c->board_size;
    L.Gpad = (c->num_games + kTile - 1) / kTile * kTile;
    L.stats_off = align256((size_t)(L.Gpad / 32 * chunk_state_bytes((int)C)));
    L.total = L.stats_off + align256((size_t)kStatStripes * 8 * 8);
    return L;
}

typedef int (*tile_fn)(const hexb_env *, const Params &, cudaStream_t);
typedef int (*sample_fn)(const View &, int, const double *, int32_t *, cudaStream_t);
typedef int (*import_fn)(const Params &, const int8_t *, const int8_t *, const uint8_t *, cudaStream_t);
#define X(n) hexb_launch_tile_##n,
static const tile_fn k_tile[] = {HEXB_FOR_N(X)};
#undef X
#define X(n) hexb_launch_sample_##n,
static const sample_fn k_sample[] = {HEXB_FOR_N(X)};
#undef X
#define X(n) hexb_launch_import_##n,
static const import_fn k_import[] = {HEXB_FOR_N(X)};
#undef X
typedef int (*mcts_fn)(int, const View &, const MctsArgs &, cudaStream_t);
#define X(n) hexb_launch_mcts_##n,
static const mcts_fn k_mcts[] = {HEXB_FOR_N(X)};
#undef X
typedef int (*playouts_fn)(const View &, const PlayoutArgs &, cudaStream_t);
#define X(n) hexb_launch_playouts_##n,
static const playouts_fn k_playouts[] = {HEXB_FOR_N(X)};
#undef X

static int dispatch_tile(const hexb_env *e, const Params &P, cudaStream_t s) {
    const int n = e->cfg.board_size;
    if (n < HEXB_MIN_BOARD || n > HEXB_MAX_BOARD) return HEXB_ERR_ARG;
    return k_tile[n - HEXB_MIN_BOARD](e, P, s);
}

static View view_of(const hexb_env *e) {
    View V;
    V.state = e->base.state;
    V.G = e->base.G;
    V.Gpad = e->base.Gpad;
    V.N = e->cfg.board_size;
    V.variant = e->cfg.variant;
    V.raw = e->cfg.raw;
    V.obs_f32 = e->base.obs_f32;
    return V;
}

// hexb_hostpack.cpp (host only): 2-bit codes -> obs + mask bytes on a pool of host threads
extern "C" HEXB_LOCAL void hexb_hostpack_expand(const uint32_t *packed, long long first_word, long long n_words, long long n_cells,
                                                int variant, int8_t *obs, uint8_t *mask);
extern "C" HEXB_LOCAL int hexb_hostpack_threads(void);
extern "C" HEXB_LOCAL void hexb_hostpack_begin(const uint32_t *packed, long long first_word, long long n_words, long long n_cells, int variant,
                                                int8_t *obs, uint8_t *mask);
extern "C" HEXB_LOCAL void hexb_hostpack_publish(long long words_arrived_abs);
extern "C" HEXB_LOCAL void hexb_hostpack_finish(int abort);

extern "C" {

int32_t hexb_version(void) { return (1 << 16) | 5; }   // 1.3: obs_dtype, launch forms, hexb_gae, packed / asynchronous host step (+ hexb_mem_alloc: additive); 1.4: hexb_set_eval, hexb_set_opponent_eps; 1.5: hexb_copy_games, hexb_playouts

const char *hexb_strerror(int32_t code) {
    switch (code) {
        case HEXB_OK: return "ok";
        case HEXB_ERR_ARG: return "bad argument or unsupported configuration";
        case HEXB_ERR_CUDA: return "CUDA call failed";
        case HEXB_ERR_STATE: return "state buffer too small or misaligned";
        case HEXB_ERR_NOGPU: return "no usable CUDA device";
        default: return "unknown error";
    }
}

int32_t hexb_last_cuda_error(void) { return g_last_cuda; }

size_t hexb_state_bytes(const hexb_config *cfg) { return cfg_ok(cfg) ? layout_of(cfg).total : 0; }

int32_t hexb_create(const hexb_config *cfg, void *state, size_t state_bytes, void *stream, hexb_env **out) {
    if (!cfg_ok(cfg) || !out) return HEXB_ERR_ARG;
    const Layout L = layout_of(cfg);
    if (!state || state_bytes < L.total || ((uintptr_t)state & 255)) return HEXB_ERR_STATE;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev) return HEXB_ERR_NOGPU;
    CK(cudaSetDevice(cfg->device));
    CK(cudaMemsetAsync(state, 0, L.total, (cudaStream_t)stream));
    hexb_env *e = (hexb_env *)calloc(1, sizeof(hexb_env));
    if (!e) return HEXB_ERR_ARG;
    e->cfg = *cfg;
    Params &P = e->base;
    P.state = (uint8_t *)state;
    P.stats = (long long *)((uint8_t *)state + L.stats_off);
    P.G = cfg->num_games;
    P.Gpad = L.Gpad;
    P.game_offset = cfg->game_offset;
    P.seed = cfg->seed;
    P.variant = cfg->variant;
    P.auto_reset = cfg->auto_reset;
    P.eval_state = cfg->eval_state;
    P.opponent_first = cfg->opponent_first;
    P.agent_mode = cfg->agent_mode;
    P.raw = cfg->raw;
    P.manual_opponent = cfg->manual_opponent;
    P.pool_size = cfg->pool_size;
    P.obs_f32 = cfg->obs_dtype == HEXB_OBS_F32 ? 1 : 0;
    P.opp_eps = -1.0;
    P.one = 1u;
    {   // L2 policy of the chunk copies (see l2_policy): when the packed state is too large to live in L2 anyway, keep a fixed
        // 20 MiB of it there across steps and stream the rest. Measured on 11x11: 1 Mi games 99.4 -> 93.0 us per step,
        // 768 Ki 76.2 -> 70.6, 2 Mi 191.2 -> 182.7; 16-24 MiB is the optimum (32: 94.1, 48: 97.2, everything: 99.6 us - the L2
        // holds only so many evict_last lines before they thrash among themselves); below ~64 MiB of state it does not pay.
        const long long cb = chunk_state_bytes(cfg->board_size * cfg->board_size);
        const long long state = L.Gpad / 32 * cb;
        P.keep_chunks = state > (64ll << 20) ? (20ll << 20) / cb : 0;
        enc_consts(P.variant, P.enc_ka, P.enc_kb, P.enc_kc);
    }
    {   // host-buffer step: adaptive DMA / packed split unless HEXB_HOST_DMA_FRACTION pins it (1 = plain DMA only)
        const char *hf = getenv("HEXB_HOST_DMA_FRACTION");
        e->host_dma_frac = 0.5;
        if (hf) {
            const double f = atof(hf);
            if (f >= 0.0 && f <= 1.0) { e->host_dma_frac = f; e->host_frac_fixed = 1; }
        }
        if (hexb_hostpack_threads() < 1) { e->host_dma_frac = 1.0; e->host_frac_fixed = 1; }
    }
    *out = e;
    return HEXB_OK;
}

int32_t hexb_destroy(hexb_env *env) {
    if (!env) return HEXB_ERR_ARG;
    if (env->host_ev || env->host_packed) cudaSetDevice(env->cfg.device);
    if (env->host_ev) {
        cudaEventDestroy(env->host_ev);
        cudaEventDestroy(env->host_ev_dma0);
        for (int k = 0; k < HEXB_HOST_SLICES; ++k) cudaEventDestroy(env->host_ev_slice[k]);
    }
    if (env->host_packed) cudaFreeHost(env->host_packed);
    free(env);
    return HEXB_OK;
}

int32_t hexb_get_config(const hexb_env *env, hexb_config *out) {
    if (!env || !out) return HEXB_ERR_ARG;
    *out = env->cfg;
    return HEXB_OK;
}

int32_t hexb_set_launch_form(hexb_env *env, int32_t warps_per_chunk) {
    if (!env || !(warps_per_chunk == 0 || warps_per_chunk == 1 || warps_per_chunk == 4)) return HEXB_ERR_ARG;
    env->launch_form = warps_per_chunk;
    return HEXB_OK;
}

int32_t hexb_set_info_buffers(hexb_env *env, int32_t *last_move_opponent, int8_t *winner) {
    if (!env) return HEXB_ERR_ARG;
    env->base.info_opp = last_move_opponent;
    env->base.info_winner = winner;
    return HEXB_OK;
}

int32_t hexb_set_opponent_buffers(hexb_env *env, int32_t *opp_index, uint8_t *to_move) {
    if (!env) return HEXB_ERR_ARG;
    env->base.opp_index = opp_index;
    env->base.to_move = to_move;
    return HEXB_OK;
}

int32_t hexb_set_eval(hexb_env *env, int32_t eval_state, int32_t *eval_episode, void *stream) {
    if (!env || env->cfg.variant != HEXB_VARIANT_B || env->cfg.raw) return HEXB_ERR_ARG;
    if (eval_episode) {
        CK(cudaSetDevice(env->cfg.device));
        CK(cudaMemsetAsync(eval_episode, 0, sizeof(int32_t) * (size_t)env->base.G, (cudaStream_t)stream));
    }
    env->cfg.eval_state = env->base.eval_state = eval_state ? 1 : 0;
    env->base.eval_episode = eval_episode;
    return HEXB_OK;
}

int32_t hexb_set_opponent_eps(hexb_env *env, double eps) {
    if (!env || env->cfg.variant != HEXB_VARIANT_A || !env->cfg.manual_opponent || !(eps == eps)) return HEXB_ERR_ARG;
    env->base.opp_eps = eps < 0.0 ? -1.0 : eps;
    return HEXB_OK;
}

int32_t hexb_half_step(hexb_env *env, int32_t side, const int32_t *actions, float *reward, uint8_t *done, void *term_obs,
                       void *stream) {
    // actions == null is allowed for side 1 only: the built-in random opponent moves (positions imported with the opponent to move)
    if (!env || env->cfg.raw || (side != 0 && side != 1) || (!actions && side != 1)) return HEXB_ERR_ARG;
    if (!env->cfg.manual_opponent) return HEXB_ERR_ARG;   // fused handles step with hexb_step; their resets already open
    CK(cudaSetDevice(env->cfg.device));
    Params P = env->base;
    P.mode = MODE_HALF;
    P.half_side = side;
    P.actions = actions;
    P.reward = reward;
    P.done = done;
    P.term_obs = (int8_t *)term_obs;
    return dispatch_tile(env, P, (cudaStream_t)stream);
}

int32_t hexb_reset(hexb_env *env, const uint8_t *reset_mask, const double *open_u, void *obs, uint8_t *mask, void *stream) {
    if (!env) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    Params P = env->base;
    P.mode = MODE_RESET;
    P.reset_mask = reset_mask;
    P.open_u = open_u;
    P.obs = (int8_t *)obs;
    P.mask = mask;
    return dispatch_tile(env, P, (cudaStream_t)stream);
}

int32_t hexb_step(hexb_env *env, const int32_t *actions, const double *opp_u, void *obs, uint8_t *mask, float *reward,
                  uint8_t *done, void *term_obs, int32_t *actions_out, void *stream) {
    if (!env || env->cfg.raw || env->cfg.manual_opponent) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    Params P = env->base;
    P.mode = MODE_STEP;
    P.steps = 1;
    P.actions = actions;
    P.opp_u = opp_u;
    P.obs = (int8_t *)obs;
    P.mask = mask;
    P.reward = reward;
    P.done = done;
    P.term_obs = (int8_t *)term_obs;
    P.actions_out = actions_out;
    return dispatch_tile(env, P, (cudaStream_t)stream);
}

int32_t hexb_rollout(hexb_env *env, int32_t num_steps, void *obs, uint8_t *mask, float *reward, uint8_t *done, void *term_obs,
                     int32_t *actions_out, void *stream) {
    if (!env || env->cfg.raw || env->cfg.manual_opponent || num_steps < 1 || num_steps > 65536) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    Params P = env->base;
    P.mode = MODE_STEP;
    P.steps = num_steps;
    P.obs = (int8_t *)obs;
    P.mask = mask;
    P.reward = reward;
    P.done = done;
    P.term_obs = (int8_t *)term_obs;
    P.actions_out = actions_out;
    return dispatch_tile(env, P, (cudaStream_t)stream);
}

// ---- the step with HOST buffers
static size_t obs_elem(const hexb_env *env) { return env->base.obs_f32 ? 4 : 1; }

size_t hexb_host_workspace_bytes(const hexb_config *cfg) {
    if (!cfg_ok(cfg)) return 0;
    const size_t G = (size_t)cfg->num_games, C = (size_t)cfg->board_size * cfg->board_size;
    const size_t ob = cfg->obs_dtype == HEXB_OBS_F32 ? 4 : 1;
    // actions | obs | mask | reward | done | packed observation words (hexb_step_host_packed)
    return align256(G * 4) + align256(G * C * ob + 16) + align256(G * C) + align256(G * 4) + align256(G) + align256((G * C + 15) / 16 * 4);
}

struct HostWs {
    int32_t *act;
    uint8_t *obs, *mask;
    float *rew;
    uint8_t *done;
    uint32_t *packed;
};
static HostWs carve_ws(const hexb_env *env, void *workspace) {
    const size_t G = (size_t)env->cfg.num_games, C = (size_t)env->cfg.board_size * env->cfg.board_size;
    uint8_t *w = (uint8_t *)workspace;
    HostWs h;
    h.act = (int32_t *)w;       w += align256(G * 4);
    h.obs = w;                  w += align256(G * C * obs_elem(env) + 16);
    h.mask = w;                 w += align256(G * C);
    h.rew = (float *)w;         w += align256(G * 4);
    h.done = w;                 w += align256(G);
    h.packed = (uint32_t *)w;
    return h;
}

// How the observation + mask bytes of a host-buffer step travel. They are 2*N*N of the 2*N*N + 5 bytes per game a step returns,
// and on the boxes this was measured on the device->host DMA path (~53 GB/s for one GPU, ~95 GB/s for all eight GPUs of a VM
// together) and the host cores' own store bandwidth (~50 GB/s on 16 cores, ~130 GB/s on 32) are separate bottlenecks. So the
// games of a step are split: the first `dma_games` games' obs / mask rows are copied as they are, the others cross PCIe as
// 2 bits per cell (K10) and host threads expand them into the same arrays (hexb_hostpack.cpp) while the DMA runs. The split
// adapts from call to call (host_step_finish); the bytes that arrive are identical for every split.
struct HostPlan {
    long long dma_games;      // games [0, dma_games) by DMA, [dma_games, G) packed
    long long first_word;     // first packed word (16 cells each) of the packed part
    long long words;          // number of packed words
};
static HostPlan plan_host(const hexb_env *env, double frac) {
    const long long G = env->cfg.num_games, C = (long long)env->cfg.board_size * env->cfg.board_size;
    HostPlan p;
    long long gd = (long long)(frac * (double)G + 0.5);
    gd = gd / 32 * 32;              // 32*C cells: a multiple of 16, so the packed part starts on a word (and 32-byte) boundary
    if (gd > G) gd = G;
    if (frac >= 1.0) gd = G;
    if (gd < 0) gd = 0;
    p.dma_games = gd;
    p.first_word = gd * C / 16;
    p.words = (G * C + 15) / 16 - p.first_word;
    if (gd == G) p.words = 0;
    return p;
}

// The packed words travel in kHostSlices pieces of growing size (cumulative 64ths below): nothing can be expanded before the
// first piece has arrived, so it is small (1/64 of the words: about 10 us of PCIe time for 1 Mi games of 11x11), and since the
// host pool works on one job per step (hexb_hostpack_begin / _publish / _finish) the pieces only set how early words become
// available, not how often the threads have to meet.
enum { kHostSlices = HEXB_HOST_SLICES };
static const int kSliceCum[kHostSlices + 1] = {0, 1, 4, 12, 24, 40, 64};

static int host_events(hexb_env *env) {
    if (env->host_ev) return HEXB_OK;
    CK(cudaEventCreateWithFlags(&env->host_ev, cudaEventDefault));
    CK(cudaEventCreateWithFlags(&env->host_ev_dma0, cudaEventDefault));
    for (int k = 0; k < kHostSlices; ++k) CK(cudaEventCreateWithFlags(&env->host_ev_slice[k], cudaEventDisableTiming));
    return HEXB_OK;
}

// Enqueue one host-buffer step. frac = share of the games whose obs / mask rows travel by DMA (1 = all, 0 = all packed).
static int host_step_enqueue(hexb_env *env, void *workspace, uint32_t *packed_host, double frac, const int32_t *actions_host,
                             void *obs_host, uint8_t *mask_host, float *reward_host, uint8_t *done_host, cudaStream_t s) {
    const long long G = env->cfg.num_games, C = (long long)env->cfg.board_size * env->cfg.board_size;
    const HostWs h = carve_ws(env, workspace);
    const size_t ob = obs_elem(env);
    CK(cudaSetDevice(env->cfg.device));
    int rc = host_events(env);
    if (rc != HEXB_OK) return rc;
    const bool can_pack = packed_host && obs_host && mask_host && !env->base.obs_f32;
    const HostPlan p = plan_host(env, can_pack ? frac : 1.0);
    if (actions_host) CK(cudaMemcpyAsync(h.act, actions_host, (size_t)G * 4, cudaMemcpyHostToDevice, s));
    const bool need_mask_dev = mask_host && p.dma_games > 0;
    rc = hexb_step(env, actions_host ? h.act : nullptr, nullptr, obs_host ? h.obs : nullptr, need_mask_dev ? h.mask : nullptr,
                   reward_host ? h.rew : nullptr, done_host ? h.done : nullptr, nullptr, nullptr, (void *)s);
    if (rc != HEXB_OK) return rc;
    env->host_plan_words = p.words;
    env->host_plan_first = p.first_word;
    if (p.words > 0) {
        // the packed words first (they are small): host threads expand slice k while the later copies are still in flight
        hexb_pack_obs_kernel<<<(unsigned)((p.words + 255) / 256), 256, 0, s>>>(reinterpret_cast<const uint4 *>(h.obs) + p.first_word, p.words,
                                                                            h.packed + p.first_word);
        CK(cudaGetLastError());
        for (int k = 0; k < kHostSlices; ++k) {
            long long lo = p.first_word + ((p.words * kSliceCum[k] / 64) & ~15ll), hi = p.first_word + ((p.words * kSliceCum[k + 1] / 64) & ~15ll);
            if (k == kHostSlices - 1) hi = p.first_word + p.words;
            env->host_slice_lo[k] = lo;
            env->host_slice_hi[k] = hi;
            if (hi > lo) CK(cudaMemcpyAsync(packed_host + lo, h.packed + lo, (size_t)(hi - lo) * 4, cudaMemcpyDeviceToHost, s));
            CK(cudaEventRecord(env->host_ev_slice[k], s));
        }
    }
    CK(cudaEventRecord(env->host_ev_dma0, s));
    const size_t dma_cells = (size_t)(p.dma_games * C);
    if (obs_host && dma_cells) CK(cudaMemcpyAsync(obs_host, h.obs, dma_cells * ob, cudaMemcpyDeviceToHost, s));
    if (mask_host && dma_cells) CK(cudaMemcpyAsync(mask_host, h.mask, dma_cells, cudaMemcpyDeviceToHost, s));
    if (reward_host) CK(cudaMemcpyAsync(reward_host, h.rew, (size_t)G * 4, cudaMemcpyDeviceToHost, s));
    if (done_host) CK(cudaMemcpyAsync(done_host, h.done, (size_t)G, cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(env->host_ev, s));
    env->host_dma_bytes = (double)dma_cells * (double)(ob + 1);
    env->host_packed_src = packed_host;
    env->host_obs = (int8_t *)obs_host;
    env->host_mask = mask_host;
    env->host_pending = 1;
    return HEXB_OK;
}

static double now_ms() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return 1e3 * (double)ts.tv_sec + 1e-6 * (double)ts.tv_nsec;
}

// Adaptive split of the host transport. The two paths are not independent - on a box where several GPUs copy at once they
// share the host's memory system, and plain DMA bytes turned out more expensive there than host-written ones (8 GPUs: all packed
// 15.1 ms, 34 % DMA 18.4 ms, all DMA 22 ms per step; one GPU: 6.3 / 4.2 (60 % DMA) / 5.1 ms) - so balancing two measured rates
// finds the wrong split, and a hill climb on single call durations random-walks on their noise (both were tried, profiles/README).
// What is robust is a small tournament: after one throw-away call (it allocates the staging), five coarse splits are timed three
// times each in rotation, the best median wins, its two neighbours at +-0.125 are timed the same way, and the winner stays.
// 22 calls in all; the search restarts every 8,192 calls in case the box's load has changed.
static const double kCoarse[5] = {0.0, 0.25, 0.5, 0.75, 0.97};
static const double kTuneMargin = 0.92;   // a split replaces the incumbent only if its median is at least 8 % shorter
static double median3(const double *v) {
    const double a = v[0], b = v[1], c = v[2];
    return a > b ? (b > c ? b : (a > c ? c : a)) : (a > c ? a : (b > c ? c : b));
}
static double tune_candidate(const hexb_env *env, int k) {   // k-th split of the running search (0..4 coarse, 5..6 fine)
    if (k < 5) return kCoarse[k];
    const double f = env->host_tune_best + (k == 5 ? -0.125 : 0.125);
    return f < 0.0 ? 0.0 : (f > 0.97 ? 0.97 : f);
}
static void tune_next(hexb_env *env, double ms) {
    int &n = env->host_tune_calls;
    if (n == 0) {                       // throw-away call done: start the coarse round
        n = 1;
        env->host_dma_frac = kCoarse[0];
        return;
    }
    if (n <= 15) {                      // coarse: call n measured candidate (n-1) % 5, sample (n-1) / 5
        env->host_tune_ms[(n - 1) % 5][(n - 1) / 5] = ms;
        if (n == 15) {
            // candidate 0 (everything packed) is the incumbent: it moves the least data over the device->host path the GPUs of a
            // box share, so its time depends least on what the other ranks happen to be trying at that moment. A split has to beat
            // the incumbent by kTuneMargin to replace it (8 ranks, r2r: the plain argmin of 3-call medians settled on 37.5 % DMA =
            // 16.2 ms per step on a box where all-packed takes 14.3 ms).
            int best = 0;
            for (int k = 1; k < 5; ++k)
                if (median3(env->host_tune_ms[k]) < kTuneMargin * median3(env->host_tune_ms[best])) best = k;
            env->host_tune_best = kCoarse[best];
            env->host_tune_best_ms = median3(env->host_tune_ms[best]);
        }
        ++n;
        env->host_dma_frac = n <= 15 ? kCoarse[(n - 1) % 5] : tune_candidate(env, 5);
        return;
    }
    if (n <= 21) {                      // fine: call n measured candidate 5 + (n-16) % 2, sample (n-16) / 2
        env->host_tune_ms[5 + (n - 16) % 2][(n - 16) / 2] = ms;
        if (n == 21) {
            double f = env->host_tune_best, t = env->host_tune_best_ms;
            for (int k = 5; k < 7; ++k)
                if (median3(env->host_tune_ms[k]) < kTuneMargin * t) { t = median3(env->host_tune_ms[k]); f = tune_candidate(env, k); }
            env->host_dma_frac = f;     // settled
            ++n;
            return;
        }
        ++n;
        env->host_dma_frac = tune_candidate(env, 5 + (n - 16) % 2);
        return;
    }
    if (++n > 22 + 8192) n = 1, env->host_dma_frac = kCoarse[0];   // search again after a while
}

// Finish the pending step: expand the packed slices as they arrive, wait for the DMA part, and (adaptive mode) feed the search.
static int host_step_finish(hexb_env *env, bool adapt) {
    env->host_pending = 0;
    CK(cudaSetDevice(env->cfg.device));
    const long long cells = (long long)env->cfg.num_games * env->cfg.board_size * env->cfg.board_size;
    if (env->host_plan_words > 0) {
        // the pool gets the whole range at once and works on it while the pieces arrive: this thread waits for each piece's copy and
        // publishes how far the words are there, then works along; one join per step (hexb_hostpack.cpp)
        hexb_hostpack_begin(env->host_packed_src, env->host_plan_first, env->host_plan_words, cells, env->cfg.variant, env->host_obs,
                            env->host_mask);
        cudaError_t err = cudaSuccess;
        for (int k = 0; k < kHostSlices && err == cudaSuccess; ++k) {
            err = cudaEventSynchronize(env->host_ev_slice[k]);
            if (err == cudaSuccess) hexb_hostpack_publish(env->host_slice_hi[k]);
        }
        hexb_hostpack_finish(err != cudaSuccess);   // always: it releases the pool
        if (err != cudaSuccess) return hexb_cuda_fail(err);
    }
    CK(cudaEventSynchronize(env->host_ev));
    if (adapt) tune_next(env, now_ms() - env->host_t0_ms);
    return HEXB_OK;
}

static int host_staging(hexb_env *env) {   // pinned staging for the packed words, owned by the handle
    if (env->host_packed) return HEXB_OK;
    CK(cudaSetDevice(env->cfg.device));
    CK(cudaHostAlloc((void **)&env->host_packed, hexb_host_packed_bytes(&env->cfg) + 64, cudaHostAllocDefault));
    return HEXB_OK;
}

int32_t hexb_step_host_begin(hexb_env *env, void *workspace, const int32_t *actions_host, void *obs_host, uint8_t *mask_host,
                             float *reward_host, uint8_t *done_host, void *stream) {
    if (!env || !workspace || env->cfg.raw || env->cfg.manual_opponent || env->host_pending) return HEXB_ERR_ARG;
    // the hybrid transport needs both arrays, int8 observations, a host thread pool and enough games to split
    const bool hybrid = obs_host && mask_host && !env->base.obs_f32 && env->host_dma_frac < 1.0 && env->cfg.num_games >= 4096;
    if (hybrid) {
        const int rc = host_staging(env);
        if (rc != HEXB_OK) return rc;
    }
    env->host_adapt = hybrid && env->host_frac_fixed == 0;
    env->host_t0_ms = now_ms();
    return host_step_enqueue(env, workspace, hybrid ? env->host_packed : nullptr, env->host_dma_frac, actions_host, obs_host, mask_host,
                             reward_host, done_host, (cudaStream_t)stream);
}

int32_t hexb_step_host_end(hexb_env *env) {
    if (!env || !env->host_pending) return HEXB_ERR_ARG;
    return host_step_finish(env, false);   // the caller's own work sits between _begin and _end: the duration says nothing about the split
}

int32_t hexb_step_host(hexb_env *env, void *workspace, const int32_t *actions_host, void *obs_host, uint8_t *mask_host,
                       float *reward_host, uint8_t *done_host, void *stream) {
    const int rc = hexb_step_host_begin(env, workspace, actions_host, obs_host, mask_host, reward_host, done_host, stream);
    if (rc != HEXB_OK) return rc;
    if (!env->host_pending) return HEXB_ERR_ARG;
    return host_step_finish(env, env->host_adapt != 0);
}

int32_t hexb_set_host_transport(hexb_env *env, double dma_fraction) {
    if (!env || env->host_pending) return HEXB_ERR_ARG;
    if (dma_fraction < 0.0) {            // adaptive (the default)
        env->host_frac_fixed = 0;
        env->host_dma_frac = 0.5;
        env->host_tune_calls = 0;
    } else {
        if (dma_fraction > 1.0) return HEXB_ERR_ARG;
        env->host_frac_fixed = 1;
        env->host_dma_frac = dma_fraction;
    }
    return HEXB_OK;
}

int32_t hexb_get_host_transport(const hexb_env *env, double *dma_fraction) {
    if (!env || !dma_fraction) return HEXB_ERR_ARG;
    *dma_fraction = env->host_dma_frac;
    return HEXB_OK;
}

int32_t hexb_step_host_packed(hexb_env *env, void *workspace, void *packed_host, const int32_t *actions_host, int8_t *obs_host,
                              uint8_t *mask_host, float *reward_host, uint8_t *done_host, void *stream) {
    if (!env || !workspace || !packed_host || env->cfg.raw || env->cfg.manual_opponent || env->host_pending) return HEXB_ERR_ARG;
    if (env->base.obs_f32 || !obs_host || !mask_host) return HEXB_ERR_ARG;   // the transport carries int8 observations; the mask is implied
    const int rc = host_step_enqueue(env, workspace, (uint32_t *)packed_host, 0.0, actions_host, obs_host, mask_host, reward_host, done_host,
                                     (cudaStream_t)stream);
    if (rc != HEXB_OK) return rc;
    return host_step_finish(env, false);
}

size_t hexb_host_packed_bytes(const hexb_config *cfg) {
    if (!cfg_ok(cfg)) return 0;
    const size_t cells = (size_t)cfg->num_games * cfg->board_size * cfg->board_size;
    return (cells + 15) / 16 * 4;
}

int32_t hexb_host_threads(void) { return hexb_hostpack_threads(); }

// ---- hexb_mem_alloc / hexb_mem_free: virtual-memory-management allocations whose physical memory may be compressible. The
// driver entry points are resolved at run time (cudaGetDriverEntryPoint), so libhexb.so has no link-time dependency on libcuda.
namespace {
struct DrvApi {
    CUresult (*GetGranularity)(size_t *, const CUmemAllocationProp *, CUmemAllocationGranularity_flags);
    CUresult (*Create)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *, unsigned long long);
    CUresult (*GetProps)(CUmemAllocationProp *, CUmemGenericAllocationHandle);
    CUresult (*Reserve)(CUdeviceptr *, size_t, size_t, CUdeviceptr, unsigned long long);
    CUresult (*Map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long);
    CUresult (*SetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t);
    CUresult (*Unmap)(CUdeviceptr, size_t);
    CUresult (*AddressFree)(CUdeviceptr, size_t);
    CUresult (*Release)(CUmemGenericAllocationHandle);
    bool ok;
};
const DrvApi &drv() {
    static const DrvApi api = [] {
        DrvApi a = {};
        const char *names[9] = {"cuMemGetAllocationGranularity", "cuMemCreate", "cuMemGetAllocationPropertiesFromHandle", "cuMemAddressReserve",
                                "cuMemMap", "cuMemSetAccess", "cuMemUnmap", "cuMemAddressFree", "cuMemRelease"};
        void **slots[9] = {(void **)&a.GetGranularity, (void **)&a.Create, (void **)&a.GetProps, (void **)&a.Reserve, (void **)&a.Map,
                           (void **)&a.SetAccess, (void **)&a.Unmap, (void **)&a.AddressFree, (void **)&a.Release};
        a.ok = true;
        for (int i = 0; i < 9; ++i) {
            cudaDriverEntryPointQueryResult st;
            if (cudaGetDriverEntryPoint(names[i], slots[i], cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess || !*slots[i])
                a.ok = false;
        }
        return a;
    }();
    return api;
}
struct MemRec {
    CUmemGenericAllocationHandle handle;
    size_t size;
    int device;
};
std::map<CUdeviceptr, MemRec> g_mem;
std::mutex g_mem_mu;
}  // namespace

int32_t hexb_mem_alloc(int32_t device, size_t bytes, int32_t compressible, void **ptr, int32_t *granted) {
    if (!ptr || bytes == 0) return HEXB_ERR_ARG;
    *ptr = nullptr;
    if (granted) *granted = 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return HEXB_ERR_NOGPU;
    int prev_dev = -1;
    cudaGetDevice(&prev_dev);
    struct Restore {   // the caller's current device is left as it was
        int dev;
        ~Restore() { if (dev >= 0) cudaSetDevice(dev); }
    } restore{prev_dev};
    CK(cudaSetDevice(device));
    CK(cudaFree(nullptr));   // the device's primary context exists and is current: the driver calls below use it
    const DrvApi &d = drv();
    if (!d.ok) return HEXB_ERR_CUDA;
    for (int attempt = compressible ? 0 : 1; attempt < 2; ++attempt) {   // compressible first, ordinary memory if the driver refuses
        CUmemAllocationProp prop = {};
        prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
        prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
        prop.location.id = device;
        prop.allocFlags.compressionType = attempt == 0 ? CU_MEM_ALLOCATION_COMP_GENERIC : CU_MEM_ALLOCATION_COMP_NONE;
        size_t gran = 0;
        if (d.GetGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0) continue;
        const size_t size = (bytes + gran - 1) / gran * gran;
        CUmemGenericAllocationHandle h;
        if (d.Create(&h, size, &prop, 0) != CUDA_SUCCESS) continue;
        CUmemAllocationProp got = {};
        const bool comp = d.GetProps(&got, h) == CUDA_SUCCESS && got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC;
        CUdeviceptr p = 0;
        if (d.Reserve(&p, size, 0, 0, 0) != CUDA_SUCCESS) { d.Release(h); continue; }
        if (d.Map(p, size, 0, h, 0) != CUDA_SUCCESS) { d.AddressFree(p, size); d.Release(h); continue; }
        CUmemAccessDesc acc = {};
        acc.location = prop.location;
        acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        if (d.SetAccess(p, size, &acc, 1) != CUDA_SUCCESS) { d.Unmap(p, size); d.AddressFree(p, size); d.Release(h); continue; }
        {
            std::lock_guard<std::mutex> lock(g_mem_mu);
            g_mem[p] = MemRec{h, size, device};
        }
        *ptr = (void *)p;
        if (granted) *granted = comp ? 1 : 0;
        return HEXB_OK;
    }
    return HEXB_ERR_CUDA;
}

int32_t hexb_mem_free(void *ptr) {
    if (!ptr) return HEXB_OK;
    MemRec r;
    {
        std::lock_guard<std::mutex> lock(g_mem_mu);
        auto it = g_mem.find((CUdeviceptr)ptr);
        if (it == g_mem.end()) return HEXB_ERR_ARG;
        r = it->second;
        g_mem.erase(it);
    }
    const DrvApi &d = drv();
    if (!d.ok) return HEXB_ERR_CUDA;
    int prev_dev = -1;
    cudaGetDevice(&prev_dev);
    cudaSetDevice(r.device);
    cudaDeviceSynchronize();   // nothing may still be using the range
    d.Unmap((CUdeviceptr)ptr, r.size);
    d.AddressFree((CUdeviceptr)ptr, r.size);
    d.Release(r.handle);
    if (prev_dev >= 0) cudaSetDevice(prev_dev);
    return HEXB_OK;
}

int32_t hexb_ply(hexb_env *env, const int32_t *actions, int8_t *ret, void *stream) {
    if (!env || !actions || !env->cfg.raw) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    Params P = env->base;
    P.mode = MODE_PLY;
    P.actions = actions;
    P.ret = ret;
    return dispatch_tile(env, P, (cudaStream_t)stream);
}

int32_t hexb_encode(hexb_env *env, int32_t view, void *obs, uint8_t *mask, void *stream) {
    if (!env || (view != 0 && view != 1)) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    const View V = view_of(env);
    const long long n = V.G * V.N * V.N;
    hexb_encode_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(V, view, (int8_t *)obs, mask);
    CK(cudaGetLastError());
    return HEXB_OK;
}

int32_t hexb_sample_actions(hexb_env *env, int32_t view, const double *u, int32_t *actions_out, void *stream) {
    if (!env || !u || !actions_out || (view != 0 && view != 1)) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    const View V = view_of(env);
    return k_sample[V.N - HEXB_MIN_BOARD](V, view, u, actions_out, (cudaStream_t)stream);
}

int32_t hexb_export_state(hexb_env *env, double *board, double *regions, double *region_counter, int8_t *cur, uint8_t *done,
                          int8_t *winner, int8_t *agent, uint32_t *draws, void *stream) {
    if (!env) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    const View V = view_of(env);
    const long long n = V.G * 2 * (V.N + 2) * (V.N + 2);
    hexb_export_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(V, board, regions, region_counter, cur, done, winner,
                                                                                       agent, draws);
    CK(cudaGetLastError());
    return HEXB_OK;
}

int32_t hexb_import_boards(hexb_env *env, const int8_t *board_true, const int8_t *to_move, const uint8_t *import_mask, void *stream) {
    if (!env || !board_true) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    return k_import[env->cfg.board_size - HEXB_MIN_BOARD](env->base, board_true, to_move, import_mask, (cudaStream_t)stream);
}

int32_t hexb_import_labels(hexb_env *env, const int8_t *board_true, const uint8_t *regions, const int8_t *to_move,
                           const uint8_t *import_mask, void *stream) {
    if (!env || !board_true || !regions) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    const Params P = env->base;
    hexb_import_labels_kernel<<<(unsigned)((P.G + 127) / 128), 128, 0, (cudaStream_t)stream>>>(P, env->cfg.board_size, board_true, regions,
                                                                                                to_move, import_mask);
    CK(cudaGetLastError());
    return HEXB_OK;
}

int32_t hexb_copy_games(hexb_env *dst, const hexb_env *src, const int64_t *src_index, const int64_t *dst_index, int64_t count,
                        void *stream) {
    if (!dst || !src || !dst->cfg.raw || count < 0) return HEXB_ERR_ARG;
    if (dst->cfg.board_size != src->cfg.board_size || dst->cfg.variant != src->cfg.variant || dst->cfg.device != src->cfg.device)
        return HEXB_ERR_ARG;
    if (count == 0) return HEXB_OK;
    CK(cudaSetDevice(dst->cfg.device));
    CopyArgs A;
    A.dst = dst->base.state;
    A.src = src->base.state;
    A.dst_G = dst->base.G;
    A.src_G = src->base.G;
    A.count = count;
    A.src_index = src_index;
    A.dst_index = dst_index;
    A.N = dst->cfg.board_size;
    hexb_copy_kernel<<<(unsigned)((count + 3) / 4), 128, 0, (cudaStream_t)stream>>>(A);
    CK(cudaGetLastError());
    return HEXB_OK;
}

int32_t hexb_playouts(hexb_env *env, int32_t num_playouts, int64_t first_playout, const uint8_t *game_mask, int32_t *wins,
                      void *stream) {
    if (!env || !wins || num_playouts < 1 || first_playout < 0 || first_playout + (int64_t)num_playouts >= (1ll << 32)) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    const View V = view_of(env);
    PlayoutArgs A;
    A.seed = env->base.seed;
    A.game_offset = (unsigned long long)env->base.game_offset;
    A.first = first_playout;
    A.num = num_playouts;
    A.game_mask = game_mask;
    A.wins = wins;
    return k_playouts[V.N - HEXB_MIN_BOARD](V, A, (cudaStream_t)stream);
}

// ---- tree search (hexb_mcts.cuh). The host checks the arguments; the kernels check the tree header init wrote, so that no
// call on a buffer that holds no tree of this handle writes anything.
static bool mcts_buffer_ok(const void *tree, size_t tree_bytes) { return tree && tree_bytes >= 128 && ((uintptr_t)tree & 15) == 0; }

static MctsArgs mcts_args(const hexb_env *env, const void *tree, size_t tree_bytes) {
    MctsArgs A;
    memset(&A, 0, sizeof(A));
    A.tree = (uint8_t *)tree;
    A.tree_bytes = tree_bytes;
    A.seed = env->base.seed;
    A.game_offset = (unsigned long long)env->base.game_offset;
    return A;
}

static int mcts_launch(const hexb_env *env, int op, const MctsArgs &A, void *stream) {
    CK(cudaSetDevice(env->cfg.device));
    const View V = view_of(env);
    return k_mcts[V.N - HEXB_MIN_BOARD](op, V, A, (cudaStream_t)stream);
}

int32_t hexb_mcts_tree_bytes(const hexb_env *env, int32_t max_nodes, size_t *bytes) {
    if (!env || !bytes || max_nodes < 1 || max_nodes > kMctsMaxNodes) return HEXB_ERR_ARG;
    const unsigned long long root = (unsigned long long)mc_root_bytes(env->cfg.board_size, max_nodes);
    const unsigned long long G = (unsigned long long)env->base.G;
    if (root > (SIZE_MAX - 128) / G) return HEXB_ERR_ARG;
    *bytes = (size_t)(128 + root * G);
    return HEXB_OK;
}

int32_t hexb_mcts_init(const hexb_env *env, void *tree, size_t tree_bytes, int32_t max_nodes, double c_puct, double fpu,
                       int64_t first_playout, const uint8_t *root_mask, void *stream) {
    size_t need = 0;
    if (!env || hexb_mcts_tree_bytes(env, max_nodes, &need) != HEXB_OK) return HEXB_ERR_ARG;
    if (!(c_puct == c_puct) || !(fpu == fpu) || first_playout < 0 || first_playout >= (1ll << 32)) return HEXB_ERR_ARG;
    if (!mcts_buffer_ok(tree, tree_bytes) || tree_bytes < need) return HEXB_ERR_STATE;
    MctsArgs A = mcts_args(env, tree, tree_bytes);
    A.max_nodes = max_nodes;
    A.c_puct = (float)c_puct;
    A.fpu = (float)fpu;
    A.first_playout = first_playout;
    A.root_mask = root_mask;
    return mcts_launch(env, MCTS_INIT, A, stream);
}

int32_t hexb_mcts_search(const hexb_env *env, void *tree, size_t tree_bytes, int32_t num_simulations, int32_t playouts_per_leaf,
                         void *stream) {
    if (!env || num_simulations < 1 || playouts_per_leaf < 1 || playouts_per_leaf > kMctsMaxPlayouts) return HEXB_ERR_ARG;
    if (!mcts_buffer_ok(tree, tree_bytes)) return HEXB_ERR_STATE;
    MctsArgs A = mcts_args(env, tree, tree_bytes);
    A.sims = num_simulations;
    A.playouts = playouts_per_leaf;
    return mcts_launch(env, MCTS_SEARCH, A, stream);
}

int32_t hexb_mcts_select(const hexb_env *env, void *tree, size_t tree_bytes, void *leaf_obs, uint8_t *leaf_mask, uint8_t *pending,
                         void *stream) {
    if (!env || !leaf_obs || !leaf_mask || !pending) return HEXB_ERR_ARG;
    if (!mcts_buffer_ok(tree, tree_bytes)) return HEXB_ERR_STATE;
    MctsArgs A = mcts_args(env, tree, tree_bytes);
    A.leaf_obs = leaf_obs;
    A.leaf_mask = leaf_mask;
    A.pending = pending;
    return mcts_launch(env, MCTS_SELECT, A, stream);
}

int32_t hexb_mcts_expand(const hexb_env *env, void *tree, size_t tree_bytes, const float *priors, const float *values, void *stream) {
    if (!env || !priors || !values) return HEXB_ERR_ARG;
    if (!mcts_buffer_ok(tree, tree_bytes)) return HEXB_ERR_STATE;
    MctsArgs A = mcts_args(env, tree, tree_bytes);
    A.priors = priors;
    A.values = values;
    return mcts_launch(env, MCTS_EXPAND, A, stream);
}

int32_t hexb_mcts_root(const hexb_env *env, const void *tree, size_t tree_bytes, int32_t *visits, float *q, float *value,
                       int32_t *nodes_used, void *stream) {
    if (!env) return HEXB_ERR_ARG;
    if (!mcts_buffer_ok(tree, tree_bytes)) return HEXB_ERR_STATE;
    MctsArgs A = mcts_args(env, tree, tree_bytes);
    A.visits = visits;
    A.q = q;
    A.value = value;
    A.nodes_used = nodes_used;
    return mcts_launch(env, MCTS_ROOT, A, stream);
}

int32_t hexb_mcts_advance(const hexb_env *env, void *tree, size_t tree_bytes, int64_t first_playout, const uint8_t *root_mask,
                          void *stream) {
    if (!env || first_playout < 0 || first_playout >= (1ll << 32)) return HEXB_ERR_ARG;
    if (!mcts_buffer_ok(tree, tree_bytes)) return HEXB_ERR_STATE;
    MctsArgs A = mcts_args(env, tree, tree_bytes);
    A.first_playout = first_playout;
    A.root_mask = root_mask;
    return mcts_launch(env, MCTS_ADVANCE, A, stream);
}

int32_t hexb_stats(hexb_env *env, int64_t *out8, void *stream) {
    if (!env || !out8) return HEXB_ERR_ARG;
    CK(cudaSetDevice(env->cfg.device));
    hexb_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(env->base.stats, out8);
    CK(cudaGetLastError());
    return HEXB_OK;
}

int32_t hexb_masked_sample(const float *logits, const uint8_t *mask, const double *u, int64_t num_games, int32_t num_cells,
                           int32_t *actions, float *logp, float *entropy, int32_t device, void *stream) {
    if (!logits || !mask || !u || num_games < 1 || num_cells < 1 || num_cells > HEXB_MAX_BOARD * HEXB_MAX_BOARD) return HEXB_ERR_ARG;
    CK(cudaSetDevice(device));
    const unsigned grid = (unsigned)((num_games * 32 + 127) / 128);
    hexb_masked_sample_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(logits, mask, u, num_games, num_cells, actions, logp, entropy);
    CK(cudaGetLastError());
    return HEXB_OK;
}

int32_t hexb_gae(const float *rewards, const float *values, const uint8_t *dones, int32_t num_steps, int64_t num_games, double gamma,
                 double gae_lambda, float *advantages, float *returns, int32_t device, void *stream) {
    if (!rewards || !values || !dones || !advantages || num_steps < 1 || num_games < 1) return HEXB_ERR_ARG;
    CK(cudaSetDevice(device));
    // gamma * lambda is formed in double like the Python expression `self.gamma * self.gae_lambda * nonterminal` it replaces
    const float gl = (float)(gamma * gae_lambda);
    hexb_gae_kernel<<<(unsigned)((num_games + 127) / 128), 128, 0, (cudaStream_t)stream>>>(rewards, values, dones, num_steps, num_games,
                                                                                            (float)gamma, gl, advantages, returns);
    CK(cudaGetLastError());
    return HEXB_OK;
}

}  // extern "C"
