// TEST INFRASTRUCTURE ONLY - host-side emulator of the CUDA kernels.
//
// Compiles the SAME device code the kernels run (hex_gym_env_b200/csrc/hexb_phases.cuh, hexb_views.cuh, hexb_search.cuh,
// hexb_mcts.cuh) with HEXB_HOST_EMU. The step kernel is replayed one warp (chunk of 32 games) at a time: every phase is run for
// all 32 "lanes" before the next one, which is what the __syncwarp() between phases guarantees on the GPU. In the copy and
// playout kernels a warp's ballot becomes a loop over its 32 lanes, and in the tree search the warp becomes one lane that owns
// every cell and every path entry, so its shuffles become loops. The extern "C" entries mirror the device's launchers
// (hexb_step_inst.cu, hexb_kernels.cu) and are driven through ctypes by tests/emu/emu.py. It lets the CPU test-suite check the
// device logic against the oracle in a container without a GPU. It is not a CPU fallback: the product package never loads it,
// and it is far too slow to be one.
#define HEXB_HOST_EMU 1
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>
#include <vector>

#include "../../hex_gym_env_b200/csrc/hexb_mcts.cuh"

using namespace hexb;

struct emu_env {
    int N;
    Params base;
    std::vector<uint8_t> state;
};

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Which relabel sweep to replay: the device picks the batched form (several rows per warp pass) for single steps of at most
// one wave of warps and for rollouts, the one-row-per-pass form for deeper launches and for reset / ply / half step.
// -1 = like the device for a small batch, 0 / 1 = force one form (so that CPU tests cover both).
static int g_force_sweep = -1;

template <int N>
static void run_tiles(Params P) {
    constexpr int C = Geo<N>::C;
    std::vector<uint8_t> smem(Geo<N>::CHUNK_STATE + 16);
    uint8_t *chunk = smem.data() + ((16 - ((uintptr_t)smem.data() & 15)) & 15);
    std::vector<Rec<N>> recs(kWarp);
    std::vector<Loc> locs(kWarp);
    uint32_t prmA[kWarp], prmB[kWarp], flg[kWarp];
    const int steps = P.mode == MODE_STEP ? P.steps : 1;
    for (long long g0 = 0; g0 < P.Gpad; g0 += kWarp) {   // one "warp" = one chunk of 32 games at a time
        uint8_t *gl = P.state + (g0 / kWarp) * Geo<N>::CHUNK_STATE;
        memcpy(chunk, gl, Geo<N>::CHUNK_STATE);
        uint32_t *recw = reinterpret_cast<uint32_t *>(chunk + Geo<N>::CHUNK_LAB);
        for (int t = 0; t < kWarp; ++t) load_rec<N>(recw + t, recs[t]);
        for (int st = 0; st < steps; ++st) {   // hexb_rollout: several env steps on the resident chunk
            const long long so = (long long)st * P.G;
            for (int t = 0; t < kWarp; ++t) {   // thread-per-game phase
                const long long g = g0 + t;
                uint8_t *L = chunk + t * C;
                prmA[t] = prmB[t] = flg[t] = 0;
                if (P.mode == MODE_STEP) {
                    double ua = 0.0, uo = 0.0;
                    if (g < P.G) pre_draws(P, recs[t].meta, recs[t].draws, (unsigned long long)(P.game_offset + g), ua, uo);
                    game_step<N>(L, P, g, st, recs[t], ua, uo, locs[t], prmA[t], prmB[t], flg[t]);
                    for (int i = 0; i < 8; ++i) P.stats[i] += locs[t].st[i];
                } else if (P.mode == MODE_RESET) {
                    game_reset<N>(P, g, recs[t], flg[t]);
                } else if (P.mode == MODE_HALF) {
                    game_half<N>(L, P, g, recs[t], locs[t], prmA[t], prmB[t], flg[t]);
                    for (int i = 0; i < 8; ++i) P.stats[i] += locs[t].st[i];
                } else {
                    game_ply<N>(L, P, g, recs[t], prmA[t], flg[t]);
                }
            }
            for (int r = 0; r < kWarp; ++r) {   // warp-per-game row jobs; a lane-level barrier = finish the loop over lanes
                if (!(flg[r] & F_ROWJOB)) continue;
                if (flg[r] & F_TERM)
                    for (int lane = 0; lane < kWarp; ++lane) term_row_lane<N>(chunk, r, flg[r], P, g0 + r + so, lane);
                for (int lane = 0; lane < kWarp; ++lane)
                    row_job_lane<N>(chunk, r, flg[r] & ~F_TERM, P, g0 + r + so, lane, [] {});
            }
            const bool batched = g_force_sweep < 0 ? (P.mode == MODE_STEP) : (g_force_sweep != 0);
            if (!batched) {
                for (int pass = 0; pass < 2; ++pass)   // like the device: rows with a single (old -> new) pair first, then the others
                    for (int r = 0; r < kWarp; ++r)
                        if ((flg[r] & (F_RELABEL | F_RESET)) == F_RELABEL) {
                            RelabelReq q;
                            prep_request(prmA[r], prmB[r], q);
                            if ((q.nx != 0u) != (pass == 1)) continue;
                            for (int lane = 0; lane < kWarp; ++lane) {
                                if (pass == 0) relabel_row_lane2<N, false>(reinterpret_cast<uint32_t *>(chunk), row_desc<N>(r), lane, q.so0, q.sn0, 0u, 0u, 0, 1u);
                                else relabel_row_lane2<N, true>(reinterpret_cast<uint32_t *>(chunk), row_desc<N>(r), lane, q.so0, q.sn0, q.xo, q.xn, (int)q.nx, 1u);
                            }
                        }
            } else {   // batched relabel sweeps, as the device kernel runs them: lane group sg takes the sg-th pending row of a parity class
                using SW = Sweep<N>;
                uint32_t olds[kWarp], news[kWarp], cnt[kWarp], pend_all = 0;
                for (int r = 0; r < kWarp; ++r) {
                    olds[r] = news[r] = cnt[r] = 0;
                    if ((flg[r] & (F_RELABEL | F_RESET)) == F_RELABEL) {
                        canon_request(prmA[r], prmB[r], olds[r], news[r], cnt[r]);
                        pend_all |= 1u << r;
                    }
                }
                const int classes = (Chunk<N>::ALIGNED_ROWS || SW::RPS == 1) ? 1 : 2;
                for (int cls = 0; cls < classes; ++cls) {
                    uint32_t pp = classes == 1 ? pend_all : (pend_all & (cls ? 0xaaaaaaaau : 0x55555555u));
                    while (pp) {
                        uint32_t next = pp;
                        for (int lane = 0; lane < kWarp; ++lane) {
                            uint32_t q = pp;
                            const int row = pick_row<N>(q, lane / SW::LPR);
                            next = q;
                            relabel_rows_lane<N>(reinterpret_cast<uint32_t *>(chunk), row, lane % SW::LPR, olds[row & 31], news[row & 31],
                                                 row >= 0 ? (int)cnt[row] : 0, 1u);
                        }
                        pp = next;
                    }
                }
            }
            if (P.mode != MODE_PLY && P.mode != MODE_HALF && (P.obs || P.mask)) {   // elementwise encode, then the rare opponent-view rows
                const long long out0 = (g0 + so) * C, limit = (so + P.G) * C;
                for (int i = 0; i < Chunk<N>::VECS; ++i) {
                    Vec4 in, o, m;
                    memcpy(&in, chunk + 16 * i, 16);
                    encode_vec<N>(in, P.variant, o, m);
                    if (P.obs) store_tail(reinterpret_cast<uint8_t *>(P.obs), out0 + 16ll * i, limit, o);
                    if (P.mask) store_tail(P.mask, out0 + 16ll * i, limit, m);
                }
                for (int r = 0; r < kWarp; ++r)
                    if (flg[r] & F_VIEW_OPP)
                        for (int lane = 0; lane < kWarp; ++lane) view_row_lane<N>(chunk, r, P, g0 + r + so, lane);
            }
        }
        for (int t = 0; t < kWarp; ++t)
            if (g0 + t < P.G) store_rec<N>(recw + t, recs[t]);
        memcpy(gl, chunk, Geo<N>::CHUNK_STATE);
    }
}

// f(std::integral_constant<int, N>()) for the board size N, as the device's per-N launcher tables pick hexb_launch_*_<n>
template <class F>
static void for_board(int N, F &&f) {
    switch (N) {
#define X(n) \
    case n: f(std::integral_constant<int, n>()); break;
        X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19)
#undef X
    }
}

static void dispatch(const emu_env *e, const Params &P) {
    for_board(e->N, [&](auto n) { run_tiles<n>(P); });
}

static View view_of(const emu_env *e) {
    View V;
    V.state = e->base.state;
    V.G = e->base.G;
    V.Gpad = e->base.Gpad;
    V.N = e->N;
    V.variant = e->base.variant;
    V.raw = e->base.raw;
    V.obs_f32 = 0;
    return V;
}

// hexb_playout_kernel<N, POLICY>: one "warp" per game, its lanes' playouts one after another
template <int N, int POLICY>
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
            won += playout_winner<N, POLICY>(black, empty, to_move, A.seed, A.game_offset + (unsigned long long)g, (uint32_t)(A.first + j),
                                             -1) == to_move;
        A.wins[g] = won;
    }
}

// hexb_mcts_*_kernel<N>: op and policy as hexb_launch_mcts_<n> takes them; the tree buffer is host memory
template <int N>
static void mcts_n(int op, int policy, const View &V, const MctsArgs &A) {
    if (op == MCTS_INIT) {
        mc_write_header(A, N, V.G);
        for (long long g = 0; g < V.G; ++g) mc_init_root<N>(V, A, g);
        return;
    }
    Tree T;
    if (!mc_tree(A, N, V.G, T)) return;
    if (op == MCTS_ADVANCE) mc_write_first_playout(A);
    for (long long g = 0; g < V.G; ++g) switch (op) {
            case MCTS_SEARCH:
                if (policy == PLAYOUT_BRIDGE) mc_search_root<N, PLAYOUT_BRIDGE>(T, A, V.variant, g);
                else mc_search_root<N, PLAYOUT_RANDOM>(T, A, V.variant, g);
                break;
            case MCTS_SELECT: mc_select_root<N>(T, V, A, g); break;
            case MCTS_EXPAND: mc_expand_root<N>(T, V, A, g); break;
            case MCTS_ROOT: mc_root_out(T, V.variant, A, g); break;
            case MCTS_ADVANCE: mc_advance_root<N>(T, V, A, g); break;
        }
}

extern "C" {

void *emu_create(int N, int variant, long long G, long long game_offset, unsigned long long seed, int agent_mode, int opponent_first,
                 int auto_reset, int eval_state, int raw) {
    if (N < 3 || N > 19 || G < 1) return nullptr;
    emu_env *e = new emu_env();
    e->N = N;
    const long long C = (long long)N * N;
    const long long Gpad = (G + kTile - 1) / kTile * kTile;
    const size_t stats_off = align256((size_t)(Gpad / 32 * chunk_state_bytes((int)C)));
    e->state.assign(stats_off + 256 + 256, 0);
    uint8_t *base = e->state.data();
    base += (256 - ((uintptr_t)base & 255)) & 255;
    Params &P = e->base;
    memset(&P, 0, sizeof(P));
    P.state = base;
    P.stats = (long long *)(base + stats_off);
    P.G = G; P.Gpad = Gpad; P.game_offset = game_offset; P.seed = seed;
    P.variant = variant; P.auto_reset = auto_reset; P.eval_state = eval_state; P.opponent_first = opponent_first;
    P.agent_mode = agent_mode; P.raw = raw; P.one = 1u; P.opp_eps = -1.0;
    return e;
}
void emu_destroy(void *h) { delete (emu_env *)h; }
void emu_force_sweep(int form) { g_force_sweep = form; }
void emu_set_manual_opponent(void *h, int pool_size, int32_t *opp_index, uint8_t *to_move) {
    emu_env *e = (emu_env *)h;
    e->base.manual_opponent = 1; e->base.pool_size = pool_size; e->base.opp_index = opp_index; e->base.to_move = to_move;
}
void emu_set_eval(void *h, int eval_state, int32_t *eval_episode, long long G) {   // what hexb_set_eval does (SelfPlayEnv.set_eval)
    emu_env *e = (emu_env *)h;
    e->base.eval_state = eval_state ? 1 : 0;
    e->base.eval_episode = eval_episode;
    if (eval_episode) memset(eval_episode, 0, sizeof(int32_t) * (size_t)G);
}
void emu_set_opponent_eps(void *h, double eps) { ((emu_env *)h)->base.opp_eps = eps < 0.0 ? -1.0 : eps; }   // hexb_set_opponent_eps
void emu_set_info(void *h, int32_t *opp, int8_t *winner) {
    emu_env *e = (emu_env *)h;
    e->base.info_opp = opp; e->base.info_winner = winner;
}
void emu_half_step(void *h, int side, const int32_t *actions, float *reward, uint8_t *done, int8_t *term_obs) {
    emu_env *e = (emu_env *)h;
    Params P = e->base;
    P.mode = MODE_HALF; P.half_side = side; P.actions = actions; P.reward = reward; P.done = done; P.term_obs = term_obs;
    dispatch(e, P);
}

void emu_reset(void *h, const uint8_t *reset_mask, const double *open_u, int8_t *obs, uint8_t *mask) {
    emu_env *e = (emu_env *)h;
    Params P = e->base;
    P.mode = MODE_RESET; P.reset_mask = reset_mask; P.open_u = open_u; P.obs = obs; P.mask = mask;
    dispatch(e, P);
}
void emu_step(void *h, const int32_t *actions, const double *opp_u, int8_t *obs, uint8_t *mask, float *reward, uint8_t *done,
              int8_t *term_obs, int32_t *actions_out) {
    emu_env *e = (emu_env *)h;
    Params P = e->base;
    P.mode = MODE_STEP; P.steps = 1; P.actions = actions; P.opp_u = opp_u; P.obs = obs; P.mask = mask; P.reward = reward; P.done = done;
    P.term_obs = term_obs; P.actions_out = actions_out;
    dispatch(e, P);
}
void emu_rollout(void *h, int steps, int8_t *obs, uint8_t *mask, float *reward, uint8_t *done, int8_t *term_obs, int32_t *actions_out) {
    emu_env *e = (emu_env *)h;
    Params P = e->base;
    P.mode = MODE_STEP; P.steps = steps; P.obs = obs; P.mask = mask; P.reward = reward; P.done = done;
    P.term_obs = term_obs; P.actions_out = actions_out;
    dispatch(e, P);
}
void emu_ply(void *h, const int32_t *actions, int8_t *ret) {
    emu_env *e = (emu_env *)h;
    Params P = e->base;
    P.mode = MODE_PLY; P.actions = actions; P.ret = ret;
    dispatch(e, P);
}
void emu_encode(void *h, int view, int8_t *obs, uint8_t *mask) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    for (long long i = 0; i < V.G * V.N * V.N; ++i) encode_at(V, view, i, obs, mask);
}
void emu_sample_actions(void *h, int view, const double *u, int32_t *out) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    for_board(V.N, [&](auto n) {
        for (long long g = 0; g < V.G; ++g) sample_at<n>(V, view, g, u, out);
    });
}
void emu_export_state(void *h, double *board, double *regions, double *counter, int8_t *cur, uint8_t *done, int8_t *winner,
                      int8_t *agent, uint32_t *draws) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    const long long n = V.G * 2 * (V.N + 2) * (V.N + 2);
    for (long long i = 0; i < n; ++i) export_at(V, i, board, regions, counter, cur, done, winner, agent, draws);
}
void emu_import_boards(void *h, const int8_t *board_true, const int8_t *to_move, const uint8_t *import_mask) {
    emu_env *e = (emu_env *)h;
    for_board(e->N, [&](auto n) {
        for (long long g = 0; g < e->base.G; ++g) import_game<n>(e->base, g, board_true, to_move, import_mask);
    });
}
void emu_import_labels(void *h, const int8_t *board_true, const uint8_t *planes, const int8_t *to_move, const uint8_t *import_mask) {
    emu_env *e = (emu_env *)h;
    for (long long g = 0; g < e->base.G; ++g) import_labels_game(e->base, e->N, g, board_true, planes, to_move, import_mask);
}
// the device's Philox4x32-10 and draw construction on their own (tests/test_philox.py: Random123 known-answer vectors)
void emu_philox4x32_10(const uint32_t *ctr4, const uint32_t *key2, uint32_t *out2) {
    philox4x32_10(ctr4[0], ctr4[1], ctr4[2], ctr4[3], key2[0], key2[1], out2[0], out2[1]);
}
double emu_draw01(unsigned long long seed, unsigned long long game, uint32_t idx) { return draw01(seed, game, idx); }
void emu_stats(void *h, int64_t *out8) {
    emu_env *e = (emu_env *)h;
    for (int i = 0; i < 8; ++i) out8[i] = e->base.stats[i];
}

// the step kernel's word-wise observation / mask encode (encode_word_k with the per-variant constants) and the per-byte
// definition it must agree with (encode_byte, agent's view), for tests/test_emu_parity.py
void emu_encode_word(unsigned int x, int variant, unsigned int *obs, unsigned int *msk) {
    uint32_t ka, kb, kc, o, m;
    enc_consts(variant, ka, kb, kc);
    encode_word_k(x, 1u, ka, kb, kc, o, m);
    *obs = o;
    *msk = m;
}
void emu_encode_byte(unsigned int b, int variant, unsigned int *obs, unsigned int *msk) {
    uint32_t m;
    *obs = encode_byte(b, variant, false, m) & 0xffu;
    *msk = m;
}

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

// hexb_playouts_policy (policy PLAYOUT_RANDOM or PLAYOUT_BRIDGE)
void emu_playouts(void *h, int num_playouts, long long first_playout, int policy, const uint8_t *game_mask, int32_t *wins) {
    emu_env *e = (emu_env *)h;
    const View V = view_of(e);
    PlayoutArgs A;
    A.seed = e->base.seed;
    A.game_offset = (unsigned long long)e->base.game_offset;
    A.first = first_playout;
    A.num = num_playouts;
    A.game_mask = game_mask;
    A.wins = wins;
    for_board(e->N, [&](auto n) {
        if (policy == PLAYOUT_BRIDGE) playouts_n<n, PLAYOUT_BRIDGE>(V, A);
        else playouts_n<n, PLAYOUT_RANDOM>(V, A);
    });
}

long long emu_mcts_tree_bytes(int N, long long G, int max_nodes) { return 128 + mc_root_bytes(N, max_nodes) * G; }

// every hexb_mcts_* call on a host tree buffer (op MCTS_INIT ... MCTS_ADVANCE); the arguments op does not use are ignored
void emu_mcts(void *h, int op, uint8_t *tree, long long tree_bytes, int max_nodes, double c_puct, double fpu, long long first_playout,
              const uint8_t *root_mask, int sims, int playouts, int policy, void *leaf_obs, uint8_t *leaf_mask, uint8_t *pending,
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
    for_board(e->N, [&](auto n) { mcts_n<n>(op, policy, V, A); });
}

}  // extern "C"
