// hexb_phases.cuh - the pieces of the fused step kernel.
//
// A WARP owns a CHUNK of 32 consecutive games. The chunk's label bytes (32*C contiguous, 16-byte aligned bytes, the
// same flat [game][cell] layout as the obs / mask outputs) sit in shared memory for the whole step. The step is
//
//   game_step        thread-per-game   agent ply + random-opponent ply (validity, stone, neighbour labels, merge request,
//                                      win), reward / done, episode accounting, auto-reset bookkeeping. Purely thread
//                                      local: a ply only looks at the mover's OWN labels, so the opponent's ply does not
//                                      depend on the agent's pending relabel and both requests are applied together.
//   row jobs         warp-per-game     for every game that asked for one (ballot): the lanes sweep that game's row of label
//                                      words - terminal observation + clear + opening stone when the game restarts (rare), or
//                                      the relabel of merged groups (both plies' requests in one pass), in one of two forms:
//                                      one row per pass (relabel_row_lane2, deep launches) or several rows per pass
//                                      (relabel_rows_lane, launches of at most one wave and rollouts).
//   encode_chunk     warp, elementwise label bytes -> obs + mask bytes, 16 bytes per lane per iteration, written straight
//                                      to the [G,C] outputs. Encoding depends only on emptiness and the owner bit, never
//                                      on the game index, so no per-word bookkeeping is needed.
//
// The device kernel (hexb_kernels.cu) strings these together with __ballot_sync / __shfl_sync / __syncwarp; the host
// emulator (tests/emu) runs the same functions with plain loops over lanes.
#pragma once
#include "hexb_core.cuh"

namespace hexb {

constexpr int kWarp = 32;
constexpr int kStatStripes = 128;  // episode statistics are accumulated into [kStatStripes][8] to spread the atomics

template <int N>
struct Chunk {
    static constexpr int C = N * N;
    static constexpr int BYTES = kWarp * C;   // multiple of 16
    static constexpr int WORDS = BYTES / 4;
    static constexpr int VECS = BYTES / 16;
    static constexpr bool ALIGNED_ROWS = (C % 4) == 0;
};

// per-thread values of one step
struct Loc {
    float reward;
    int action;
    int st[8];  // episode statistics increments (see hexb.h: hexb_stats)
};

// b = address of record word 0 of this game (global memory or the chunk copy in shared memory); words are kRecStride apart
template <int N>
HEXB_HD void load_rec(const uint32_t *b, Rec<N> &r) {
    constexpr int W = Geo<N>::W;
#pragma unroll
    for (int w = 0; w < W; ++w) r.occ_rm[w] = b[w * kRecStride];
    r.meta = b[W * kRecStride];
    r.draws = b[(W + 1) * kRecStride];
}
template <int N>
HEXB_HD void store_rec(uint32_t *b, const Rec<N> &r) {
    constexpr int W = Geo<N>::W;
#pragma unroll
    for (int w = 0; w < W; ++w) b[w * kRecStride] = r.occ_rm[w];
    b[W * kRecStride] = r.meta;
    b[(W + 1) * kRecStride] = r.draws;
}

// reward HexEnv.step would hand out again for an already finished variant-A game (HexGame.py:250,267-279)
HEXB_HD float stale_reward_A(uint32_t meta) {
    if (meta & M_INVALID) return -100.f;
    const uint32_t w = (meta & M_WIN_MASK) >> M_WIN_SHIFT;
    return w == 1u ? 1.f : (w == 2u ? -1.f : 0.f);
}

// The two draws a step normally consumes, computed up front (they only depend on the stream position) so that the
// device can do the Philox arithmetic while the chunk's label bytes are still in flight:
//   u_agent  BaseRandomPolicy.choose_action of the driving loop (only when actions == null)       at draws
//   u_opp    BaseRandomPolicy.choose_action / random_policy of the opponent's reply                at draws (+1 if the agent
//            drew) (+1 for the unused random.uniform of SelfplayWrapper.py:159 in variant B)
HEXB_HD void pre_draws(const Params &P, uint32_t meta, uint32_t draws, unsigned long long gid, double &u_agent, double &u_opp) {
    uint32_t idx = draws;
    u_agent = 0.0;
    u_opp = 0.0;
    if (!(meta & M_LIVE) || (meta & M_DONE)) return;
    if (!P.actions) u_agent = draw01(P.seed, gid, idx++);
    if (!P.opp_u) u_opp = draw01(P.seed, gid, idx + (P.variant == VARIANT_B ? 1u : 0u));
}

// ---------------------------------------------------------------------------------------------- one env step of one game
// SelfPlayEnv.step (SelfplayWrapper.py:174-199) -> HexEnv.step (HexSingleGame.py:233-263) + continue_game (:146-172), or
// variant-A HexEnv.step (HexGame.py:244-295) + opponent_move (:332-349); then the DummyVecEnv-style auto-reset and the
// episode counters. With actions == null the agent is BaseRandomPolicy / random_policy itself and takes one draw from the
// game's stream first, exactly like the reference loop  a = BaseRandomPolicy().choose_action(obs); env.step(a).
// L = this game's C label bytes. prmA / prmB = relabel requests of the two plies, flg = row job for the warp.
// game_step comes in two parts so that the device can run the first one while the chunk's label bytes are still in flight:
//   game_step_pre   needs the game's RECORD only (occupancy, meta): the agent's action (given, or the k-th empty cell of its
//                   draw), its validity, and - speculatively, from the occupancy as it will be - the cell of the opponent's reply
//                   (the reply depends on the agent's ply only through one occupancy bit, not on its labels; it is used only if
//                   the reply really happens, i.e. after a legal agent move that does not end the game)
//   game_step_post  the two place_stone calls on the label bytes, reward / done, accounting, auto-reset
struct Pre {
    int a, n_reply, x_reply, cell_reply;
    bool valid;
};
template <int N>
HEXB_HD void game_step_pre(const Params &P, long long g, const Rec<N> &rec, double u_agent, double u_opp, Pre &q) {
    constexpr int C = Geo<N>::C;
    q.a = -1; q.n_reply = 0; q.x_reply = 0; q.cell_reply = 0; q.valid = false;
    if (g >= P.G || !(rec.meta & M_LIVE) || (rec.meta & M_DONE)) return;
    int a;
    if (P.actions) a = P.actions[g];
    else a = select_kth_zero<N>(rec.occ_rm, choice_of(u_agent, count_empty<N>(rec.occ_rm)));
    q.a = a;
    q.valid = (unsigned)a < (unsigned)C && !test_bit<N>(rec.occ_rm, a);
    if (q.valid) {
        uint32_t occ2[Geo<N>::W];
#pragma unroll
        for (int w = 0; w < Geo<N>::W; ++w) occ2[w] = rec.occ_rm[w] | word_bit(a, w, P.one);
        const double u = P.opp_u ? P.opp_u[2 * g] : u_opp;
        q.n_reply = count_empty<N>(occ2);
        q.cell_reply = select_kth_zero_colmajor<N>(occ2, choice_of(u, q.n_reply), q.x_reply);  // k-th empty cell of the opponent's view
    }
}
template <int N>
HEXB_HD void game_step_post(uint8_t *L, const Params &P, long long g, int t, Rec<N> &rec, const Pre &q, Loc &loc,
                            uint32_t &prmA, uint32_t &prmB, uint32_t &flg) {
    const long long o = g + (long long)t * P.G;  // output slot: step t of a multi-step launch (hexb_rollout) writes row t of [T,G]
    loc.reward = 0.f;
    loc.action = -1;
#pragma unroll
    for (int i = 0; i < 8; ++i) loc.st[i] = 0;
    prmA = 0; prmB = 0; flg = 0;
    if (g >= P.G) return;
    if (!(rec.meta & M_LIVE)) {  // never reset: nothing to play
        if (P.reward) P.reward[o] = 0.f;
        if (P.done) P.done[o] = 1;
        if (P.actions_out) P.actions_out[o] = -1;
        return;
    }
    const unsigned long long gid = (unsigned long long)(P.game_offset + g);
    const bool was_done = (rec.meta & M_DONE) != 0u;
    int opp_move = -1;
    if (was_done) {
        loc.reward = P.variant == VARIANT_A ? stale_reward_A(rec.meta) : 0.f;
    } else {
        // ---- agent ply
        if (!P.actions) rec.draws++;
        const int a = q.a;
        loc.action = a;
        loc.st[6] = 1;
        if (!q.valid) {  // fast_move returns 3, state untouched; the env ends the episode (HexGame.py:252-253, HexSingleGame.py:240-241)
            rec.meta |= M_DONE | M_INVALID | M_AGENT_ENDED;
            loc.reward = P.variant == VARIANT_A ? -100.f : 0.f;
        } else {
            const bool won = place_stone<N>(L, rec, 0, a, prmA, P.one);
            loc.st[7]++;
            rec.meta ^= M_TOMOVE;
            if (won) {
                rec.meta |= M_DONE | (1u << M_WIN_SHIFT) | M_AGENT_ENDED;
                loc.reward = 1.f;
            } else if (P.variant == VARIANT_B && q.n_reply == 0) {
                rec.meta |= M_DONE | M_AGENT_ENDED;  // HexSingleGame.py:117-119 (cannot happen from an empty start)
            }
        }
        // ---- opponent ply: continue_game (SelfplayWrapper.py:146-172) / opponent_move (HexGame.py:332-349), random policy
        if (!(rec.meta & M_DONE)) {
            if (!P.opp_u) rec.draws += (P.variant == VARIANT_B) ? 2u : 1u;  // variant B: rv = random.uniform(0,1), unused (:159), then the choice
            const int n = q.n_reply, x = q.x_reply, cell = q.cell_reply;
            // (Reading the reply's neighbourhood before the agent's stone is written - stone_merge for both plies side by side,
            // stone_commit afterwards - was measured and rejected: 15.15 vs 15.00 us at 131,072 games of 11x11, 100.0 vs 98.8 at
            // 1 Mi, profiles/r2p_merge2_ab.jsonl: the reply does not always happen, and the extra live registers cost more.)
            const bool won = place_stone<N>(L, rec, 1, cell, prmB, P.one);
            // A: the env transposes the move back to the true cell (HexGame.py:341-346); B: the index in the opponent's own view
            if (P.info_opp) opp_move = P.variant == VARIANT_A ? cell : x * N + (cell - x) / N;
            loc.st[7]++;
            rec.meta ^= M_TOMOVE;
            if (won) {
                rec.meta |= M_DONE | (2u << M_WIN_SHIFT);
                loc.reward = -1.f;
            } else if (P.variant == VARIANT_B && n == 1) {
                rec.meta |= M_DONE;
            }
        }
    }
    const bool is_done = (rec.meta & M_DONE) != 0u;
    if (is_done && !was_done) {  // episode accounting (true colours)
        const uint32_t w = (rec.meta & M_WIN_MASK) >> M_WIN_SHIFT;
        const bool tr = (rec.meta & M_TRANSPOSED) != 0u;
        loc.st[0] = 1;
        loc.st[1] = (w == 1u && !tr) || (w == 2u && tr);
        loc.st[2] = (w == 2u && !tr) || (w == 1u && tr);
        loc.st[3] = (w == 1u);
        loc.st[4] = Geo<N>::C - count_empty<N>(rec.occ_rm);  // plies of the episode = stones on the board
        loc.st[5] = (rec.meta & M_INVALID) != 0u;
        if (P.term_obs) flg |= F_TERM | (((rec.meta & M_AGENT_ENDED) && P.variant == VARIANT_B) ? F_TERM_OPP : 0u);
    }
    if (P.reward) P.reward[o] = loc.reward;
    if (P.done) P.done[o] = is_done ? 1 : 0;
    if (P.actions_out) P.actions_out[o] = loc.action;
    if (P.info_opp) P.info_opp[g] = opp_move;
    if (P.info_winner) {  // HexEnv.winner (HexGame.py:251,347 / HexSingleGame.py:239): the last make_move's return value
        const uint32_t w = (rec.meta & M_WIN_MASK) >> M_WIN_SHIFT;
        const int tr = (rec.meta & M_TRANSPOSED) ? 1 : 0;
        P.info_winner[g] = (int8_t)((rec.meta & M_INVALID) ? 3 : (w == 0u ? -1 : (int)((w - 1u) ^ (uint32_t)tr)));
    }
    if (is_done) {
        if (P.auto_reset) {
            reset_game<N>(rec, P, gid, P.opp_u ? &P.opp_u[2 * g + 1] : nullptr, flg);
            if (flg & F_OPEN) loc.st[7]++;  // the opponent's opening stone is a ply of this step
        } else if ((rec.meta & M_AGENT_ENDED) && P.variant == VARIANT_B) {
            flg |= F_VIEW_OPP;
        }
    }
    if (!(flg & F_RESET) && ((prmA | prmB) & P_NEED)) flg |= F_RELABEL;
}
template <int N>
HEXB_HD void game_step(uint8_t *L, const Params &P, long long g, int t, Rec<N> &rec, double u_agent, double u_opp, Loc &loc,
                       uint32_t &prmA, uint32_t &prmB, uint32_t &flg) {
    Pre q;
    game_step_pre<N>(P, g, rec, u_agent, u_opp, q);
    game_step_post<N>(L, P, g, t, rec, q, loc, prmA, prmB, flg);
}

// ---------------------------------------------------------------------------------------------- half step (hexb_half_step)
// One ply of ONE side for every game whose turn it is, the action coming from the caller: the agent's half of
// SelfPlayEnv.step (SelfplayWrapper.py:174-176) or the opponent's half, continue_game (:146-172) with an OpponentPolicy
// (:26-35) instead of the random policy - the caller runs the opponent network on the side-to-move view (hexb_encode view 1)
// and passes its actions in the opponent's own perspective. Reward / done / statistics / auto-reset as in game_step, except
// that a restarted game whose opponent opens is left waiting for the caller's opponent (to_move = 1).
template <int N>
HEXB_HD void game_half(uint8_t *L, const Params &P, long long g, Rec<N> &rec, Loc &loc, uint32_t &prmA, uint32_t &prmB, uint32_t &flg) {
    constexpr int C = Geo<N>::C;
    loc.reward = 0.f;
    loc.action = -1;
#pragma unroll
    for (int i = 0; i < 8; ++i) loc.st[i] = 0;
    prmA = 0; prmB = 0; flg = 0;
    if (g >= P.G) return;
    if (!(rec.meta & M_LIVE)) {
        if (P.reward) P.reward[g] = 0.f;
        if (P.done) P.done[g] = 1;
        if (P.to_move) P.to_move[g] = 2;
        return;
    }
    const unsigned long long gid = (unsigned long long)(P.game_offset + g);
    const int side = P.half_side;
    const bool was_done = (rec.meta & M_DONE) != 0u;
    const bool my_turn = (((rec.meta & M_TOMOVE) != 0u) == (side != 0));
    if (!was_done && my_turn) {
        if (side != 0 && P.variant == VARIANT_B) rec.draws++;           // rv = random.uniform(0,1), unused (SelfplayWrapper.py:159)
        int a;
        bool from_caller = P.actions != nullptr;
        if (from_caller && side != 0 && P.variant == VARIANT_A && P.opp_eps >= 0.0) {
            // HexEnv.opponent_predict (HexGame.py:354-359): rv = random.uniform(0,1); rv < eps -> random_policy(state), else the model
            from_caller = !(draw01(P.seed, gid, rec.draws++) < P.opp_eps);
        }
        if (from_caller) a = P.actions[g];
        else {  // the built-in random opponent (BaseRandomPolicy / random_policy): k-th empty cell of ITS view
            const double u = draw01(P.seed, gid, rec.draws++);
            int x;
            const int cell = select_kth_zero_colmajor<N>(rec.occ_rm, choice_of(u, count_empty<N>(rec.occ_rm)), x);
            a = x * N + (cell - x) / N;   // the same cell as an index of the opponent's own view (its transpose)
        }
        loc.action = a;
        if (side == 0) loc.st[6] = 1;                                   // an env step starts with the agent's ply
        int cell = a;
        if (side != 0 && (unsigned)a < (unsigned)C) {                   // the opponent's view is the transpose of the stored board
            const int x = a / N;
            cell = (a - x * N) * N + x;
        }
        const bool valid = (unsigned)a < (unsigned)C && !test_bit<N>(rec.occ_rm, cell);
        if (!valid) {  // fast_move returns 3; HexEnv.step ends the episode for either side (HexSingleGame.py:240-241, HexGame.py:252-253)
            rec.meta |= M_DONE | M_INVALID | (side == 0 ? M_AGENT_ENDED : 0u);
            loc.reward = (P.variant == VARIANT_A && side == 0) ? -100.f : 0.f;
        } else {
            const bool won = place_stone<N>(L, rec, side, cell, side == 0 ? prmA : prmB, P.one);
            loc.st[7]++;
            rec.meta ^= M_TOMOVE;
            if (won) {
                rec.meta |= M_DONE | ((uint32_t)(side + 1) << M_WIN_SHIFT) | (side == 0 ? M_AGENT_ENDED : 0u);
                loc.reward = side == 0 ? 1.f : -1.f;
            } else if (P.variant == VARIANT_B && count_empty<N>(rec.occ_rm) == 0) {
                rec.meta |= M_DONE | (side == 0 ? M_AGENT_ENDED : 0u);
            }
        }
    } else if (was_done && P.variant == VARIANT_A && side == 0) {
        loc.reward = stale_reward_A(rec.meta);
    }
    const bool is_done = (rec.meta & M_DONE) != 0u;
    if (is_done && !was_done) {
        const uint32_t w = (rec.meta & M_WIN_MASK) >> M_WIN_SHIFT;
        const bool tr = (rec.meta & M_TRANSPOSED) != 0u;
        loc.st[0] = 1;
        loc.st[1] = (w == 1u && !tr) || (w == 2u && tr);
        loc.st[2] = (w == 2u && !tr) || (w == 1u && tr);
        loc.st[3] = (w == 1u);
        loc.st[4] = Geo<N>::C - count_empty<N>(rec.occ_rm);
        loc.st[5] = (rec.meta & M_INVALID) != 0u;
        // what step() returned: the board after invert_board, i.e. seen by the side that would move next
        if (P.term_obs) flg |= F_TERM | (((rec.meta & M_AGENT_ENDED) && P.variant == VARIANT_B) ? F_TERM_OPP : 0u);
    }
    if (P.reward) P.reward[g] = loc.reward;
    if (P.done) P.done[g] = is_done ? 1 : 0;
    if (is_done && !was_done && P.auto_reset) reset_game<N>(rec, P, gid, nullptr, flg);
    if (P.to_move) P.to_move[g] = (rec.meta & M_DONE) ? 2 : ((rec.meta & M_TOMOVE) ? 1 : 0);
    if (!(flg & F_RESET) && ((prmA | prmB) & P_NEED)) flg |= F_RELABEL;
}

// ---------------------------------------------------------------------------------------------- raw ply (hexb_ply)
// Batched HexGame.make_move: variant A in true coordinates (HexGame.py:85-111, no done guard); variant B with the action
// in the mover's perspective, as HexEnv.step feeds it (HexSingleGame.py:239, 98-106).
template <int N>
HEXB_HD void game_ply(uint8_t *L, const Params &P, long long g, Rec<N> &rec, uint32_t &prmA, uint32_t &flg) {
    constexpr int C = Geo<N>::C;
    prmA = 0; flg = 0;
    if (g >= P.G || !(rec.meta & M_LIVE)) return;
    const int a = P.actions[g];
    const int p = (rec.meta & M_TOMOVE) ? 1 : 0;
    int r = 3;
    if ((unsigned)a < (unsigned)C) {
        const int cell = (P.variant == VARIANT_B && p) ? transpose_cell<N>(a) : a;
        if (!test_bit<N>(rec.occ_rm, cell)) {
            const bool won = place_stone<N>(L, rec, p, cell, prmA, P.one);
            rec.meta ^= M_TOMOVE;
            r = -1;
            if (won) {
                rec.meta = (rec.meta & ~M_WIN_MASK) | M_DONE | ((uint32_t)(p + 1) << M_WIN_SHIFT);
                r = p;
            } else if (P.variant == VARIANT_B && count_empty<N>(rec.occ_rm) == 0) {
                rec.meta |= M_DONE;
            }
        }
    }
    if (P.ret) P.ret[g] = (int8_t)r;
    if (prmA & P_NEED) flg |= F_RELABEL;
}

// ---------------------------------------------------------------------------------------------- reset (hexb_reset)
template <int N>
HEXB_HD void game_reset(const Params &P, long long g, Rec<N> &rec, uint32_t &flg) {
    flg = 0;
    if (g >= P.G) return;
    if (!P.reset_mask || P.reset_mask[g]) {
        reset_game<N>(rec, P, (unsigned long long)(P.game_offset + g), P.open_u ? &P.open_u[g] : nullptr, flg);
    } else if ((rec.meta & M_DONE) && (rec.meta & M_AGENT_ENDED) && P.variant == VARIANT_B && !P.raw) {
        flg |= F_VIEW_OPP;
    }
    if (P.to_move) P.to_move[g] = !(rec.meta & M_LIVE) || (rec.meta & M_DONE) ? 2 : ((rec.meta & M_TOMOVE) ? 1 : 0);
}

// ---------------------------------------------------------------------------------------------- row jobs (one lane's share)
// Row r of the chunk = bytes [r*C, (r+1)*C) = words (r*C)>>2 .. ((r+1)*C-1)>>2. For odd N a row is not word aligned and its
// first / last word also holds cells of the neighbouring games: row_mask() keeps a lane's read-modify-write inside the row.
// Rows are processed one at a time by the whole warp, so neighbouring rows are never updated concurrently.
template <int N>
HEXB_HD uint32_t row_mask(int row_start, int row_end, int w) {
    if (Chunk<N>::ALIGNED_ROWS) return 0xffffffffu;
    const int lo = row_start - 4 * w;  // bytes below lo belong to the previous game
    const int hi = row_end - 4 * w;    // bytes from hi on belong to the next game
    uint32_t m = 0xffffffffu;
    if (lo > 0) m &= 0xffffffffu << (8 * lo);
    if (hi < 4) m &= 0xffffffffu >> (8 * (4 - hi));
    return m;
}

// 0x80 in every byte of y that is zero
HEXB_HD uint32_t zero_flags(uint32_t y, uint32_t one) { return ~(fma_add(y & 0x7f7f7f7fu, 0x7f7f7f7fu, one) | y) & 0x80808080u; }

// words a row can span, and sweeps of 32 lanes needed to cover them
template <int N>
struct RowSpan {
    static constexpr int WORDS = (Geo<N>::C + 3) / 4 + (Chunk<N>::ALIGNED_ROWS ? 0 : 1);
    static constexpr int SWEEPS = (WORDS + kWarp - 1) / kWarp;
};

// ---- relabel sweep, one row per warp pass (the form for deep launches). Everything that depends only on the row index
// (first / last word, edge masks) comes from a per-board-size table in constant memory, and the step's relabel requests are
// prepared once per game by its own lane (thread-per-game, all lanes in parallel) instead of being decoded by every lane in
// every pass: the sweeps are the largest consumer of the ALU pipe, which bounds the step kernel in the steady state.
struct RowDesc {
    int w0;                // first word of the row's label bytes (the last one is w0 + RowLanes<N>::SPAN)
    uint32_t first, last;  // row_mask() of the first and the last word (all ones when rows are word aligned)
};
template <int N>
HEXB_HD constexpr RowDesc make_row_desc(int r) {
    constexpr int C = Geo<N>::C;
    const int rs = r * C, re = rs + C;
    return RowDesc{rs >> 2, (C % 4 == 0) ? 0xffffffffu : 0xffffffffu << (8 * (rs & 3)),
                   (C % 4 == 0) ? 0xffffffffu : 0xffffffffu >> (8 * (3 - ((re - 1) & 3)))};
}
#if defined(__CUDACC__) && !defined(HEXB_HOST_EMU)
template <int N>
struct RowTable {
    RowDesc d[kWarp];
    constexpr RowTable() : d{} {
        for (int r = 0; r < kWarp; ++r) d[r] = make_row_desc<N>(r);
    }
};
template <int N>
__constant__ RowTable<N> c_rowtab{};
#endif
template <int N>
HEXB_HD RowDesc row_desc(int r) {
#if defined(__CUDA_ARCH__)
    return c_rowtab<N>.d[r];
#else
    return make_row_desc<N>(r);
#endif
}

// A game's relabel work of one step: pair 0 (old byte -> new byte) splatted over a word, the other pairs (a second group merged
// by the same ply, the other ply's merges: the rarer cases) packed one per byte in xo / xn, nx = their number (0..3).
struct RelabelReq {
    uint32_t so0, sn0, xo, xn, nx;
};
HEXB_HD void canon_request(uint32_t prmA, uint32_t prmB, uint32_t &olds, uint32_t &news, uint32_t &n);
HEXB_HD void prep_request(uint32_t prmA, uint32_t prmB, RelabelReq &q) {
    uint32_t olds, news, n;
    canon_request(prmA, prmB, olds, news, n);
    q.so0 = splat(olds & 0xffu);
    q.sn0 = splat(news & 0xffu);
    q.xo = olds >> 8;
    q.xn = news >> 8;
    q.nx = n - 1u;
}
// Every row spans the same number of words, SPAN + 1 (C = N * N is a multiple of 4 for even N and 1 more than one for odd N, so a
// row that starts at byte offset r & 3 of its first word ends in word w0 + SPAN), so which lane holds a row's first or last word,
// and which lanes have nothing to do, depends on the lane alone: those tests do not depend on the row and are hoisted out of the
// warp's loop over rows.
template <int N>
struct RowLanes {
    static constexpr int SPAN = (Geo<N>::C + 3) / 4 - 1;
    static constexpr bool check() {
        for (int r = 0; r < kWarp; ++r)
            if (((r * Geo<N>::C + Geo<N>::C - 1) >> 2) - ((r * Geo<N>::C) >> 2) != SPAN) return false;
        return true;
    }
    static_assert(check(), "every row of a chunk spans SPAN + 1 words");
};
template <int N, bool EXTRA = true>
HEXB_HD void relabel_row_lane2(uint32_t *lab32, const RowDesc &d, int lane, uint32_t so0, uint32_t sn0, uint32_t xo, uint32_t xn, int nx,
                               uint32_t one) {
    constexpr int SPAN = RowLanes<N>::SPAN;
#pragma unroll
    for (int it = 0; it < RowSpan<N>::SWEEPS; ++it) {
        const int j = lane + it * kWarp;   // word j of the row
        if (j > SPAN) break;
        const int w = d.w0 + j;
        const uint32_t x = lab32[w];
        // bytes of the neighbouring games in the row's first / last word are blanked before the compare (labels are never 0)
        const uint32_t rm = (d.first | (j == 0 ? 0u : 0xffffffffu)) & (d.last | (j == SPAN ? 0u : 0xffffffffu));
        uint32_t mk = sign_fill(zero_flags((x & rm) ^ so0, one));
        uint32_t x2 = (x & ~mk) | (sn0 & mk);
#pragma unroll 1
        for (int p = 0; EXTRA && p < nx; ++p) {   // warp-uniform trip count; rows with a single pair are swept with EXTRA = false
            const uint32_t so = splat_byte_dyn(xo, p), sn = splat_byte_dyn(xn, p);
            mk = sign_fill(zero_flags((x2 & rm) ^ so, one));
            x2 = (x2 & ~mk) | (sn & mk);
        }
        lab32[w] = x2;   // (unconditional: a predicated store issues all the same, and the compare is one ALU op more)
    }
}

// ---- batched relabel sweep: several rows per warp pass.
// A row of label bytes spans at most RowSpan<N>::WORDS words; a group of LPR lanes takes one row, WPL words per lane, so one
// pass of the warp relabels RPS = 32 / LPR rows (4 rows of an 11x11 board, 8 of a 7x7 one) instead of one, with WPL independent
// words in flight per lane. Rows handled in the same pass must not share an edge word (odd N): the caller batches rows of equal
// parity, which are never adjacent.
template <int N>
struct Sweep {
    static constexpr int WPL = 4;
    static constexpr int NEED = (RowSpan<N>::WORDS + WPL - 1) / WPL;
    static constexpr int LPR = NEED <= 4 ? 4 : (NEED <= 8 ? 8 : (NEED <= 16 ? 16 : 32));
    static constexpr int RPS = kWarp / LPR;
};

// The step's two relabel requests (prm words of place_stone) as up to four (old byte -> new byte) pairs: olds / news hold
// pair p in byte p, n = number of pairs; unused slots repeat pair 0 (applying a pair twice is a no-op).
HEXB_HD void canon_request(uint32_t prmA, uint32_t prmB, uint32_t &olds, uint32_t &news, uint32_t &n) {
    olds = 0; news = 0; n = 0;
    const uint32_t prm[2] = {prmA, prmB};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const uint32_t o1 = prm[i] & 0xffu, o2 = (prm[i] >> 8) & 0xffu, m = (prm[i] >> 16) & 0xffu;
        if (prm[i] & P_NEED) {
            olds |= o1 << (8 * n); news |= m << (8 * n); n++;
            if (o2 != o1) { olds |= o2 << (8 * n); news |= m << (8 * n); n++; }
        }
    }
    if (n < 4u) {
        const uint32_t keep = (1u << (8 * n)) - 1u;
        olds = (olds & keep) | (splat(olds & 0xffu) & ~keep);
        news = (news & keep) | (splat(news & 0xffu) & ~keep);
    }
}

// The sg-th (0-based) lowest set bit of *pp for each of the RPS lane groups, -1 if there are fewer; clears the RPS lowest bits.
template <int N>
HEXB_HD int pick_row(uint32_t &pp, int sg) {
    int mine = -1;
#pragma unroll
    for (int k = 0; k < Sweep<N>::RPS; ++k) {
        int r = -1;
        if (pp) {
#if defined(__CUDA_ARCH__)
            r = __ffs(pp) - 1;
#else
            r = __builtin_ctz(pp);
#endif
        }
        if (k == sg) mine = r;
        pp &= pp - 1u;   // stays 0 once empty
    }
    return mine;
}

// position of the k-th (0-based) set bit of m, -1 if m has fewer (the cooperative kernel hands the k-th pending row to lane group k)
HEXB_HD int kth_set_bit32(uint32_t m, int k) {
    if (k >= popc32(m)) return -1;
    int pos = 0, c;
    c = popc32(m & 0xffffu); if (k >= c) { k -= c; pos += 16; m >>= 16; }
    c = popc32(m & 0xffu);   if (k >= c) { k -= c; pos += 8;  m >>= 8; }
    c = popc32(m & 0xfu);    if (k >= c) { k -= c; pos += 4;  m >>= 4; }
    c = popc32(m & 0x3u);    if (k >= c) { k -= c; pos += 2;  m >>= 2; }
    c = (int)(m & 1u);       if (k >= c) { pos += 1; }
    return pos;
}

// One lane's share of one pass: sub-lane sl of the group that owns `row` applies the row's n pairs to its WPL words
// (regions[regions == label] = new_region_label, HexGame.py:141-142, HexSingleGame.py:152-153, for both plies of the step).
template <int N>
HEXB_HD void relabel_rows_lane(uint32_t *lab32, int row, int sl, uint32_t olds, uint32_t news, int n, uint32_t one) {
    constexpr int C = Geo<N>::C, WPL = Sweep<N>::WPL, LPR = Sweep<N>::LPR;
    if (row < 0) return;
    const int rs = row * C, re = rs + C;
    const int w0 = rs >> 2, wl = (re - 1) >> 2;
    const uint32_t first = Chunk<N>::ALIGNED_ROWS ? 0xffffffffu : 0xffffffffu << (8 * (rs & 3));
    const uint32_t last = Chunk<N>::ALIGNED_ROWS ? 0xffffffffu : 0xffffffffu >> (8 * (3 - ((re - 1) & 3)));
    uint32_t x[WPL], y[WPL], rm[WPL];
#pragma unroll
    for (int j = 0; j < WPL; ++j) {
        const int w = w0 + sl + j * LPR;
        x[j] = w <= wl ? lab32[w] : 0u;   // a word outside the row holds nothing to relabel (labels are never 0)
        y[j] = x[j];
        rm[j] = (w == w0 ? first : 0xffffffffu) & (w == wl ? last : 0xffffffffu);
    }
    for (int p = 0; p < n; ++p) {
        const uint32_t so = splat_byte_dyn(olds, p), sn = splat_byte_dyn(news, p);
#pragma unroll
        for (int j = 0; j < WPL; ++j) {
            const uint32_t mk = sign_fill(zero_flags(y[j] ^ so, one)) & rm[j];
            y[j] = (y[j] & ~mk) | (sn & mk);
        }
    }
#pragma unroll
    for (int j = 0; j < WPL; ++j) {
        const int w = w0 + sl + j * LPR;
        if (y[j] != x[j]) lab32[w] = y[j];
    }
}

// Games that restart get an empty board (HexSingleGame.py:208-231 / HexGame.py:206-220) plus the opponent's opening stone
// when it moves first (flg bits 8-15 = its byte, 16-31 = its cell).
template <int N>
HEXB_HD void clear_row_lane(uint32_t *lab32, int r, uint32_t flg, int lane) {
    constexpr int C = Geo<N>::C;
    const int rs = r * C, re = rs + C;
    const int ob = rs + (int)(flg >> 16);  // chunk byte of the opening stone
#pragma unroll
    for (int it = 0; it < RowSpan<N>::SWEEPS; ++it) {
        const int w = (rs >> 2) + lane + it * kWarp;
        if (w > ((re - 1) >> 2)) break;
        const uint32_t rm = row_mask<N>(rs, re, w);
        uint32_t x = Chunk<N>::ALIGNED_ROWS ? 0u : (lab32[w] & ~rm);
        if ((flg & F_OPEN) && (ob >> 2) == w) x |= ((flg >> 8) & 0xffu) << (8 * (ob & 3));
        lab32[w] = x;
    }
}

// info["terminal_observation"] of a game that finished in this step: what step() itself returned, i.e. the opponent's view
// (transposed, signs swapped) when the agent's own ply ended the game (HexSingleGame.py:259-262), else the agent's view.
template <int N>
HEXB_HD void term_row_lane(const uint8_t *chunk, int r, uint32_t flg, const Params &P, long long g, int lane) {
    constexpr int C = Geo<N>::C;
    const uint8_t *Lg = chunk + r * C;
    const bool opp = (flg & F_TERM_OPP) != 0u;
    for (int c = lane; c < C; c += kWarp) {
        uint32_t mk;
        const uint32_t b = Lg[opp ? transpose_cell<N>(c) : c];
        store_obs(P.term_obs, P.obs_f32, g * C + c, encode_byte(b, P.variant, opp, mk));
    }
}

// obs + mask of a finished, not restarted game whose last ply was the agent's: the opponent's view (see term_row_lane).
template <int N>
HEXB_HD void view_row_lane(const uint8_t *chunk, int r, const Params &P, long long g, int lane) {
    constexpr int C = Geo<N>::C;
    const uint8_t *Lg = chunk + r * C;
    for (int c = lane; c < C; c += kWarp) {
        uint32_t mk;
        const uint32_t ob = encode_byte(Lg[transpose_cell<N>(c)], P.variant, true, mk);
        if (P.obs) store_obs(P.obs, P.obs_f32, g * C + c, ob);
        if (P.mask) P.mask[g * C + c] = (uint8_t)mk;
    }
}

// A finished game's row job, one lane's share: terminal observation (reads the finished board), then clear (+ opening stone);
// the caller separates the two with a warp barrier (`sync`), because different lanes read and write the same words.
template <int N, class SyncFn>
HEXB_HD void row_job_lane(uint8_t *chunk, int r, uint32_t flg, const Params &P, long long g, int lane, SyncFn sync) {
    uint32_t *lab32 = reinterpret_cast<uint32_t *>(chunk);
    if (flg & F_TERM) {
        term_row_lane<N>(chunk, r, flg, P, g, lane);
        sync();
    }
    if (flg & F_RESET) clear_row_lane<N>(lab32, r, flg, lane);
}

// ---------------------------------------------------------------------------------------------- encode (one lane's share)
// get_action_mask (HexGame.py:203-204) / legal_actions (HexSingleGame.py:205-206) and the observation the env returns (the
// live simulator.board: HexGame.py:294, HexSingleGame.py:262 after invert_board :265-271) in the agent's view = the stored
// orientation, for the whole chunk, elementwise: output byte i of the chunk depends on label byte i only.
struct Vec4 {
    uint32_t x, y, z, w;
};
HEXB_HD void store_tail(uint8_t *base, long long off, long long limit, const Vec4 &v) {
    const uint32_t a[4] = {v.x, v.y, v.z, v.w};
    for (int k = 0; k < 16; ++k)
        if (off + k < limit) base[off + k] = (uint8_t)(a[k >> 2] >> (8 * (k & 3)));
}
HEXB_HD void encode_vec_k(const Vec4 &in, uint32_t one, uint32_t ka, uint32_t kb, uint32_t kc, Vec4 &o, Vec4 &m) {
    encode_word_k(in.x, one, ka, kb, kc, o.x, m.x);
    encode_word_k(in.y, one, ka, kb, kc, o.y, m.y);
    encode_word_k(in.z, one, ka, kb, kc, o.z, m.z);
    encode_word_k(in.w, one, ka, kb, kc, o.w, m.w);
}
template <int N>
HEXB_HD void encode_vec(const Vec4 &in, int variant, Vec4 &o, Vec4 &m) {
    uint32_t ka, kb, kc;
    enc_consts(variant, ka, kb, kc);
    encode_vec_k(in, 1u, ka, kb, kc, o, m);
}

}  // namespace hexb
